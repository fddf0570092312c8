"""Host-side orchestration of the MISA forward / backward over libmmda_b200.so.

``MisaEngine`` owns the device workspace (packed activations, saved gates, head buffers) and
sequences the C-ABI kernels for one step.  It is used two ways:

* level 1 (drop-in): ``MISA.forward`` wraps ``engine.forward`` in one ``torch.autograd.Function``
  so the reference's own ``get_*_loss`` + ``loss.backward()`` (src/solver.py:163-183) work
  unchanged; autograd hands the output gradients to ``engine.backward``.
* level 2 (fused step): ``mmda_b200.trainer.FusedTrainer`` calls ``engine.forward``, the fused
  loss kernels, ``engine.backward`` and the clip+Adam kernel with no autograd in the loop.

PyTorch is used for device memory, streams and (in the trainer) ``torch.distributed`` only.
"""
from __future__ import annotations

import contextlib
from typing import Dict, Optional

import torch

from ._lib import LIB, MmdaError
from .config import ACTIVATIONS

MODS = ("t", "v", "a")
ENC = {"t": ("trnn1", "trnn2", "tlayer_norm"), "v": ("vrnn1", "vrnn2", "vlayer_norm"),
       "a": ("arnn1", "arnn2", "alayer_norm")}
PRIV_TAG = {"t": "1", "v": "1", "a": "3"}
ACT_NONE, ACT_LEAKY, ACT_SIGMOID, ACT_RELU = 0, 1, 2, 3
ACT_RRELU = ACTIVATIONS["rrelu"]
# random-number stream ids of training-mode RReLU (+ modality index): project_m, then
# discriminator_layer_1 on utt_shared_m.  The dropout sites use 1-8, BERT 200 and up.
SID_RRELU_PROJECT, SID_RRELU_DISC = 9, 12
LN_EPS = 1e-5
ATT_P = 0.1            # nn.TransformerEncoderLayer default dropout (reference src/models.py:160)
NHEAD = 2
TL = "transformer_encoder.layers.0."
# stream priorities; lower = sooner.  Measured: the three encoder chains at equal priority above
# the weight-gradient leaves 4.54 ms/step; text above the side chains 4.64; everything equal 4.60
PRIO_TEXT, PRIO_SIDE, PRIO_LEAF = -1, -1, 0
_DRYRUN = False       # tests only: exercise the host orchestration on CPU with a stubbed library


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


_HERE = object()       # Kernels.side(after=...) default: wait on the current stream


class Kernels:
    """Thin typed wrappers: torch tensors in, C-ABI calls out, on the stream ``bind_stream`` or
    ``side`` bound.  ``side`` / ``mark`` / ``wait`` are the only code that creates side streams,
    records or waits on events: one stream per (device, role), created on first use."""

    def __init__(self):
        self.stream = None
        self.launches = 0
        self.leaf_on = False            # set by the engine's backward
        self._leaf_used = {}            # leaf role -> None, in first-use order since the last join
        self._role = None               # role of the stream `side` runs on; None: the caller's
        self._streams = {}
        # torch.are_deterministic_algorithms_enabled() as the engine read it at its last forward /
        # backward: route every cross-CTA reduction to its fixed-order entry
        self.det = False
        self.buf_fn = None              # the engine's workspace allocator (MisaEngine.buf)

    def bind_stream(self):
        # the CPU dry run binds the role name, so that a stubbed library sees where launches go
        if _DRYRUN:
            self.stream = 0 if self._role is None else self._role
        else:
            self.stream = torch.cuda.current_stream().cuda_stream

    def _c(self, name, *args):
        self.launches += 1
        LIB.call(name, *args, self.stream)

    def det_ws(self, query, *args):
        """Scratch of a fixed-order reduction, sized by the entry's ``*_workspace_bytes`` query:
        one buffer per stream role, since the launches of one stream run in order."""
        nbytes = int(LIB.raw(query)(*args))
        if nbytes < 0:
            raise MmdaError(LIB.raw("mmda_last_error")().decode())
        return self.buf_fn(f"det_ws_{self._role}", max(4, (nbytes + 15) // 16 * 4))

    def _stream(self, role, priority=0, device=None):
        key = (torch.cuda.current_device() if device is None else device, role)
        st = self._streams.get(key)
        if st is None:
            st = self._streams[key] = torch.cuda.Stream(device=key[0], priority=priority)
        return st

    def mark(self, role=None):
        """Event at the current point of the current stream, or with ``role`` at the end of what
        ``side(role)`` blocks have enqueued so far.  None in the dry run."""
        if _DRYRUN:
            return None
        return (torch.cuda.current_stream() if role is None else self._stream(role)).record_event()

    def wait(self, *events):
        """Order the current stream after the events (None: nothing to wait for)."""
        events = [ev for ev in events if ev is not None]
        if events:
            cur = torch.cuda.current_stream()
            for ev in events:
                cur.wait_event(ev)

    @contextlib.contextmanager
    def side(self, role, priority=0, after=_HERE):
        """Run the block on ``role``'s stream of the current device, ordered after the current
        point of the current stream, or after the events ``after`` only.  Launches and torch
        operations in the block go to that stream; the caller's binding comes back on exit.  The
        dry run creates no stream: it runs the block inline with the role name bound."""
        prev = self._role, self.stream
        ctx = contextlib.nullcontext()
        if _DRYRUN:
            stream = role
        else:
            cur = torch.cuda.current_stream()
            st = self._stream(role, priority, cur.device_index)
            if after is _HERE:
                st.wait_stream(cur)
            else:
                for ev in after:
                    if ev is not None:
                        st.wait_event(ev)
            ctx, stream = torch.cuda.stream(st), st.cuda_stream
        try:
            with ctx:
                self._role, self.stream = role, stream
                yield
        finally:
            self._role, self.stream = prev

    # C = act(alpha * op(A) op(B) + beta*C + bias + bias2); A,B,C are 2-D views with unit inner stride
    def gemm(self, A, B, C, ta=False, tb=False, alpha=1.0, beta=0.0, bias=None, bias2=None,
             act=ACT_NONE, split_k=0, c_ilv=0):
        M, N = C.shape
        K = A.shape[0] if ta else A.shape[1]
        assert A.stride(1) == 1 and B.stride(1) == 1 and C.stride(1) == 1
        assert (A.shape[1] if ta else A.shape[0]) == M, (A.shape, C.shape, ta)
        assert (B.shape[0] if tb else B.shape[1]) == N and (B.shape[1] if tb else B.shape[0]) == K, \
            (A.shape, B.shape, C.shape, ta, tb)
        # deterministic: the entry that swaps every atomic split-K for the in-CTA one
        self._c("mmda_sgemm_det" if self.det else "mmda_sgemm", int(ta), int(tb), M, N, K, alpha,
                _ptr(A), A.stride(0), _ptr(B), B.stride(0), beta, _ptr(C), C.stride(0), _ptr(bias),
                _ptr(bias2), act, split_k, c_ilv)

    def gemm_tc(self, kind, a_mn, b_mn, M, N, K, A, B, C, alpha=1.0, bias=None, mode=0, split_k=1,
                c_ilv=0):
        """Tensor-core GEMM.  A, B = (hi, lo_or_None) 2-D operand views (unit inner stride)."""
        (Ah, Al), (Bh, Bl) = A, B
        if kind == 0 and Al is None:
            kind = 2     # A plain fp32 (split in shared memory); B plain (Bl None) or pre-split
        elif kind == 0 and Bl is None:
            raise MmdaError("gemm_tc: a pre-split A operand needs a pre-split B operand")
        if self.det and mode == 1 and split_k != 1:
            ws = self.det_ws("mmda_gemm_tc_det_workspace_bytes", kind, M, N, K, mode, split_k)
            self._c("mmda_gemm_tc_det", kind, int(a_mn), int(b_mn), M, N, K, _ptr(Ah), _ptr(Al),
                    Ah.stride(0), _ptr(Bh), _ptr(Bl), Bh.stride(0), alpha, _ptr(C), C.stride(0),
                    _ptr(bias), None, mode, split_k, c_ilv, _ptr(ws))
            return
        self._c("mmda_gemm_tc", kind, int(a_mn), int(b_mn), M, N, K, _ptr(Ah), _ptr(Al), Ah.stride(0),
                _ptr(Bh), _ptr(Bl), Bh.stride(0), alpha, _ptr(C), C.stride(0), _ptr(bias), None, mode,
                split_k, c_ilv)

    def linear(self, x, w, b, out, act=ACT_NONE, bias2=None):
        self.gemm(x, w, out, tb=True, bias=b, bias2=bias2, act=act)

    def leaf(self, fn):
        """Run fn() -- kernels whose results nothing later in the step's dependency chain reads
        (weight / bias gradients) -- on a side stream paired with the current one, ordered after
        everything enqueued so far.  `join_leaves()` orders the current stream after all of them.
        The caller guarantees the operands fn reads are not overwritten before the join."""
        if not self.leaf_on:
            fn()
            return
        role = ("leaf", self._role)
        with self.side(role, PRIO_LEAF):
            fn()
        self._leaf_used[role] = None

    def join_leaves(self):
        self.wait(*[self.mark(role) for role in self._leaf_used])
        self._leaf_used = {}

    def linear_bwd(self, dy, x, w, dw, db, dx=None, dx_beta=0.0, db2=None, dw_split=0):
        """dy: grad of the linear output (pre-activation).  dw/db accumulate (dw_split >= 2
        forces the atomic split-K path: needed when several streams accumulate into one dw).
        Only dx continues the backward chain: dw / db go to the leaf stream."""
        def wgrad():
            self.gemm(dy, x, dw, ta=True, beta=1.0, split_k=dw_split)
            if db is not None:
                self.colsum(dy, db, db2)
        self.leaf(wgrad)
        if dx is not None:
            self.gemm(dy, w, dx, beta=dx_beta, split_k=1 if dx_beta not in (0.0, 1.0) else 0)

    def colsum(self, x, out, out2=None, ilv=0):
        if self.det:
            ws = self.det_ws("mmda_colsum_det_workspace_bytes", x.shape[0], x.shape[1])
            self._c("mmda_colsum_det", _ptr(x), x.stride(0), x.shape[0], x.shape[1], _ptr(out),
                    _ptr(out2), ilv, _ptr(ws))
            return
        self._c("mmda_colsum", _ptr(x), x.stride(0), x.shape[0], x.shape[1], _ptr(out), _ptr(out2),
                ilv)

    def layernorm(self, x, res, g, b, y, mean, rstd):
        self._c("mmda_layernorm_forward", _ptr(x), x.stride(0), _ptr(res),
                0 if res is None else res.stride(0), _ptr(g), _ptr(b), _ptr(y), y.stride(0),
                _ptr(mean), _ptr(rstd), x.shape[0], x.shape[1], LN_EPS)

    def layernorm_bwd(self, dy, x, res, g, mean, rstd, dx, dg, db):
        if self.det:
            ws = self.det_ws("mmda_layernorm_backward_det_workspace_bytes", x.shape[0], x.shape[1])
            self._c("mmda_layernorm_backward_det", _ptr(dy), dy.stride(0), _ptr(x), x.stride(0),
                    _ptr(res), 0 if res is None else res.stride(0), _ptr(g), _ptr(mean), _ptr(rstd),
                    _ptr(dx), dx.stride(0), _ptr(dg), _ptr(db), x.shape[0], x.shape[1], _ptr(ws))
            return
        self._c("mmda_layernorm_backward", _ptr(dy), dy.stride(0), _ptr(x), x.stride(0), _ptr(res),
                0 if res is None else res.stride(0), _ptr(g), _ptr(mean), _ptr(rstd), _ptr(dx),
                dx.stride(0), _ptr(dg), _ptr(db), x.shape[0], x.shape[1])

    def act(self, x, act):
        self._c("mmda_act_forward", _ptr(x), x.stride(0), x.shape[0], x.shape[1], act)

    def act_bwd(self, dy, y, act):
        self._c("mmda_act_backward", _ptr(dy), dy.stride(0), _ptr(y), y.stride(0), dy.shape[0],
                dy.shape[1], act)

    def rrelu(self, x, seed, sid, seed_dev=None):
        """training-mode RReLU in place on the 2-D view x"""
        self._c("mmda_rrelu_forward", _ptr(x), _ptr(x), x.stride(0), x.shape[0], x.shape[1], seed,
                _ptr(seed_dev), sid)

    def rrelu_bwd(self, dy, y, seed, sid, seed_dev=None):
        assert dy.shape == y.shape and dy.stride(0) == y.stride(0)
        self._c("mmda_rrelu_backward", _ptr(dy), _ptr(y), y.stride(0), y.shape[0], y.shape[1], seed,
                _ptr(seed_dev), sid)

    def add(self, out, x, y=None, ax=1.0, ay=1.0):
        self._c("mmda_add2d", _ptr(out), out.stride(0), _ptr(x), x.stride(0), ax, _ptr(y),
                0 if y is None else y.stride(0), ay, out.shape[0], out.shape[1])

    def dropout(self, x, out, p, seed, sid, seed_dev=None):
        self._c("mmda_dropout", _ptr(x), _ptr(out), x.numel(), p, seed, _ptr(seed_dev), sid)


def _f32(*shape, device):
    return torch.empty(*shape, dtype=torch.float32, device=device)


class MisaEngine:
    def __init__(self, model):
        self.model = model
        self.cfg = model.config
        self.k = Kernels()
        self.k.buf_fn = self.buf
        self.ws: Dict[str, torch.Tensor] = {}
        self.ws_version = 0
        self.act_id = ACTIVATIONS[model.act_name]
        self.d = self.cfg.hidden_size
        self.NC = self.cfg.num_classes
        self.H = dict(zip(MODS, model.hidden_sizes))
        self._pack_key = None
        self.pad = None                 # (T_pad, Np) while FusedTrainer runs a padded (graph) step
        self._params = None
        self._params_ver = None
        self._dev = None
        self.seed = 0x5EED
        self.step_id = 0
        prec = getattr(self.cfg, "precision", "fp32")
        if prec not in ("fp32", "bf16"):
            raise ValueError(f"precision must be 'fp32' or 'bf16', got {prec!r}")
        # precision="bf16" selects bf16 operands for the BERT text encoder's GEMMs only (C4).  The
        # hoisted LSTM GEMMs always run 3xTF32 (fp32-accurate): a bf16 input projection moved this
        # model's text-encoder gradients by 5-15 % (measured round 1) and gained nothing once the
        # recurrence itself ran on tensor cores, so that mode was removed (DESIGN.md section 3.2).
        self.tc_kind = 0 if prec == "fp32" else 1
        # use_bert=True (SURVEY.md 8f N1): the BERT encoder runs on the hand-written kernels too
        # (mmda_b200/bert.py); its masked-mean output enters here as `utt_text` and backward()
        # returns the gradient wrt it.
        self._bert = None
        self.adversarial = not bool(getattr(self.cfg, "use_cmd_sim", True))
        self.diff_out = _DIFF_OUT + (tuple(f"domain_label_{m}" for m in MODS) if self.adversarial
                                     else ())
        self.use_bert = bool(self.cfg.use_bert)
        self.gru = getattr(model, "rnncell", "lstm") == "gru"        # models.py:39
        self.utt_dim = {m: 4 * self.H[m] for m in MODS}
        if self.use_bert:
            self.utt_dim["t"] = 768

    @property
    def bert(self):
        if self._bert is None:
            from .bert import BertEngine
            self._bert = BertEngine(self)
        return self._bert

    # ---------------------------------------------------------------- buffers -------------
    def buf(self, name, *shape, dtype=torch.float32, zero=False):
        dev = self._dev
        t = self.ws.get(name)
        n = 1
        for s in shape:
            n *= s
        if t is None or t.numel() < n or t.dtype != dtype or t.device != dev:
            if t is not None:
                # a captured CUDA graph may hold this buffer's raw pointer: replacing it (growth,
                # dtype, device) invalidates the graph; a buffer under a NEW name cannot be
                # referenced by any existing graph
                self.ws_version += 1
            # zero-filled: a padded launch (self.pad) runs row-wise kernels over rows no kernel
            # ever wrote, and those must at least hold finite values
            t = torch.zeros(max(n, 1), dtype=dtype, device=dev)
            self.ws[name] = t
        v = t[:n].view(*shape)
        if zero:
            v.zero_()
        return v

    @property
    def device(self):
        self.params()
        return self._dev

    def params(self) -> Dict[str, torch.Tensor]:
        # re-read when the module's tensors were replaced (.to(), embed.weight.data = ...)
        ver = tuple(p.data_ptr() for p in self.model.parameters())
        if self._params_ver != ver:
            self._dev = next(self.model.parameters()).device
            self._params = {n: p.data for n, p in self.model.named_parameters()
                            if not n.startswith("bertmodel.")}
            self._params_ver = ver
            for n, p in self._params.items():
                if not p.is_cuda and not _DRYRUN:
                    raise MmdaError(f"parameter {n} is on {p.device}: the MISA hot path runs on a "
                                    "B200 only (no CPU fallback); call model.to('cuda') first")
                if p.dtype != torch.float32 or not p.is_contiguous():
                    raise MmdaError(f"parameter {n} must be contiguous float32")
        return self._params

    # ---------------------------------------------------------------- packing -------------
    def _pack(self, lengths_cpu: torch.Tensor):
        """Same descending sort torch's pack_padded_sequence runs on the CPU lengths (so the
        permutation is bit-identical), then device-side batch_sizes / offsets / row maps."""
        if lengths_cpu.is_cuda:
            raise MmdaError("lengths must stay on the CPU (reference src/solver.py:149)")
        ln = lengths_cpu.to(torch.int64)
        pad = self.pad
        key = (ln.numel(), tuple(ln.tolist()), pad, self._dev)
        if key == self._pack_key:
            return self._pack_info
        if ln.numel() == 0 or int(ln.min()) <= 0:
            raise MmdaError("every sequence length must be >= 1 (pack_padded_sequence raises too)")
        ls, si = torch.sort(ln, descending=True)
        B, Tmax, N = ln.numel(), int(ls[0]), int(ln.sum())
        Np = N
        if pad is not None:
            # (T_pad, Np): every kernel of the step is launched over Np >= N packed rows and a
            # time extent of T_pad >= Tmax, so one captured graph serves all length patterns that
            # round to the same Np (FusedTrainer.step); the device-side lens / offsets / row maps
            # carry the real lengths
            if pad[0] < Tmax or pad[1] < N:
                raise MmdaError(f"pad {pad} smaller than the batch (Tmax={Tmax}, N={N})")
            Tmax, Np = pad
        host = torch.empty(2 * B, dtype=torch.int32)
        if not _DRYRUN:
            host = host.pin_memory()
        host[:B] = ls.to(torch.int32)
        host[B:] = si.to(torch.int32)
        dev = self.buf("pack_in", 2 * B, dtype=torch.int32)
        dev.copy_(host, non_blocking=True)
        bs = self.buf("batch_sizes", Tmax, dtype=torch.int32)
        off = self.buf("offsets", Tmax + 1, dtype=torch.int32)
        row_t = self.buf("row_t", Np, dtype=torch.int32)
        row_j = self.buf("row_j", Np, dtype=torch.int32)
        self.k._c("mmda_pack_build_padded", _ptr(dev[:B]), B, Tmax, N, Np, _ptr(bs), _ptr(off),
                  _ptr(row_t), _ptr(row_j))
        self._host_keepalive = host
        # N is the LAUNCH row count (= the real one unless padded); n_dev the real one, on the device
        self._pack_info = dict(B=B, Tmax=Tmax, N=Np, N_true=N, padded=Np != N, n_dev=off[Tmax:],
                               lens=dev[:B], sidx=dev[B:], bs=bs, off=off,
                               row_t=row_t, row_j=row_j, sorted_idx_cpu=si, lens_sorted_cpu=ls)
        self._pack_key = key
        return self._pack_info

    # ---------------------------------------------------------------- streams --------------
    def _fork(self, fns, text_first=False):
        """Run fns[m]() on modality m's stream, all after everything enqueued so far on the
        current stream, in the order v, a, t (t, v, a with ``text_first``, so that the side
        streams can wait on launch points the text function marked); join before returning.
        The text encoder is the critical path: its stream's priority places its kernels ahead of
        the visual / acoustic CTAs competing for SMs."""
        k = self.k
        start, done = k.mark(), []
        for m in (("t", "v", "a") if text_first else ("v", "a", "t")):
            with k.side(m, PRIO_TEXT if m == "t" else PRIO_SIDE, after=(start,)):
                fns[m]()
            done.append(k.mark(m))
        k.wait(*done)

    # ---------------------------------------------------------------- tensor-core operands --
    def pbuf(self, name, rows, cols):
        """(rows, cols) view of a workspace buffer whose row pitch is cols rounded up to 4 floats.
        The hoisted LSTM GEMMs run on tcgen05 for every hidden size: operands whose natural pitch
        breaks TMA's 16-byte rule (visual 35 / 70, acoustic 74 floats) live in such buffers; the
        pad columns are never read (the tensor maps carry the true extents)."""
        ld = (cols + 3) // 4 * 4
        return self.buf(name, rows, ld)[:, :cols]

    def _prep(self, name, x, out=None, row0=0, kind=None, split=False):
        """Tensor-core operand of the 2-D view x.  3xTF32 (kind 0): activations are consumed as
        plain fp32 (returned as is, the kernel splits them in shared memory); ``split=True`` makes
        the ahead-of-time (hi, lo) tf32 split -- used for weights (B operands), which every tile
        re-reads.  bf16 (kind 1, BERT encoder): a bf16 copy; rows land at [row0, row0+rows) of
        the (possibly larger) buffer `out`."""
        kind = self.tc_kind if kind is None else kind
        rows, cols = x.shape
        if kind == 0 and split:
            hi, lo = self._prep_buf(name, rows, cols, 0, split=True)
            self.k._c("mmda_split_tf32", _ptr(x), x.stride(0), rows, cols, _ptr(hi), _ptr(lo),
                      hi.stride(0))
            return hi, lo
        if kind == 0:
            if out is None and x.stride(1) == 1 and x.stride(0) % 4 == 0 and x.data_ptr() % 16 == 0:
                return x, None           # consumed as is
            raise MmdaError(f"operand {name}: 3xTF32 operands must be 16-byte aligned fp32 views")
        if out is None:
            out = self._prep_buf(name, rows, cols, kind)
        hi, lo = out
        self.k._c("mmda_cast_bf16", _ptr(x), x.stride(0), rows, cols, _ptr(hi[row0:]), hi.stride(0))
        return out

    def _prep_buf(self, name, rows, cols, kind=None, split=False):
        kind = self.tc_kind if kind is None else kind
        if kind == 0:
            ld = (cols + 3) // 4 * 4
            hi = self.buf(name + "_hi", rows, ld)[:, :cols]
            if not split:
                return hi, None
            lo = self.buf(name + "_lo", rows, ld)[:, :cols]
            return hi, lo
        ld = (cols + 7) // 8 * 8
        return self.buf(name + "_bf", rows, ld, dtype=torch.bfloat16)[:, :cols], None

    def _pack_weights(self, r, P, H, I):
        """Stacked gate-interleaved copy of layer r's W_ih (both directions), split into tf32
        hi/lo for the 3xTF32 GEMMs, + the bias stack."""
        W = self._prep_buf(f"tcW_{r}", 8 * H, I, 0, split=True)
        bst = self.buf(f"bst_{r}", 8 * H)
        self.k._c("mmda_lstm_pack_weights", _ptr(P[f"{r}.weight_ih_l0"]),
                  _ptr(P[f"{r}.weight_ih_l0_reverse"]), _ptr(P[f"{r}.bias_ih_l0"]),
                  _ptr(P[f"{r}.bias_hh_l0"]), _ptr(P[f"{r}.bias_ih_l0_reverse"]),
                  _ptr(P[f"{r}.bias_hh_l0_reverse"]), H, I, _ptr(W[0]), _ptr(W[1]),
                  W[0].stride(0), _ptr(bst))
        return W, bst

    _RNN_KEYS = ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")

    def _gru_overlay(self, m, P, what):
        """nn.GRU cells (models.py:39): 4-slot stand-ins for modality m's (3H, .) GRU tensors so
        the LSTM-shaped machinery (gate layout [N][2][H][4], stacked GEMMs) applies unchanged.
        what = "expand": build the 4-slot weights from P; "weights": the same buffers, no launch;
        "grads": zeroed 4-slot gradient buffers."""
        H = self.H[m]
        r1, r2, _ = ENC[m]
        out = {}
        for r, I in ((r1, H), (r2, 2 * H)):
            for suf in ("", "_reverse"):
                tag = "gruG" if what == "grads" else "gruW"
                shapes = ((4 * H, I), (4 * H, H), (4 * H,), (4 * H,))
                t = [self.buf(f"{tag}{i}_{r}{suf}", *sh) for i, sh in enumerate(shapes)]
                if what == "expand":
                    src = [P[f"{r}.{kk}{suf}"] for kk in self._RNN_KEYS]
                    self.k._c("mmda_gru_expand_weights", *[_ptr(x) for x in src], H, I,
                              *[_ptr(x) for x in t])
                for kk, x in zip(self._RNN_KEYS, t):
                    out[f"{r}.{kk}{suf}"] = x
        return out

    # ---- dense layers big enough for the tensor-core path (the fusion layer's FFN) ----
    def _tc_lin_ok(self, M, N, K):
        return M >= 512 and N % 4 == 0 and K % 4 == 0

    def tc_linear(self, tag, x, w, b, out):
        """out = x w^T + b on tcgen05 (3xTF32: fp32-accurate in either precision mode)."""
        M, K = x.shape
        N = w.shape[0]
        xo, wo = self._prep(tag + "_x", x, kind=0), self._prep(tag + "_w", w, kind=0, split=True)
        self.k.gemm_tc(0, 0, 0, M, N, K, xo, wo, out, bias=b)

    def tc_linear_bwd(self, tag, dy, x, w, dw, db, dx, dx_acc):
        """dw += dy^T x, db += colsum(dy), dx (+)= dy w   (dy: [M][N], x: [M][K], w: [N][K])"""
        M, N = dy.shape
        K = x.shape[1]
        dyo = self._prep(tag + "_dy", dy, kind=0)
        xo = self._prep(tag + "_x", x, kind=0)

        def wgrad():
            self.k.gemm_tc(0, 1, 1, N, K, M, dyo, xo, dw, mode=1, split_k=0)
            self.k.colsum(dy, db)
        self.k.leaf(wgrad)
        self.k.gemm_tc(0, 0, 1, M, K, N, dyo, self._prep(tag + "_w", w, kind=0, split=True), dx,
                       mode=1 if dx_acc else 0, split_k=0 if dx_acc else 1)

    @staticmethod
    def _cols(op, lo, hi):
        return (op[0][:, lo:hi], None if op[1] is None else op[1][:, lo:hi])

    def _lstm_tc_ws(self, m, B, H, Tmax):
        """Workspace of the tensor-core recurrence for modality m, or None when that path does
        not cover (B, H) -- small hidden sizes and GRU cells stay on the SIMT kernels."""
        if self.gru or _DRYRUN:
            return None
        nbytes = LIB.raw("mmda_lstm_tc_workspace_bytes")(B, H, Tmax)
        if nbytes <= 0:
            return None
        name, n = f"lstm_tc_ws_{m}", (nbytes + 3) // 4
        old = self.ws.get(name)
        ws = self.buf(name, n, dtype=torch.int32)
        if old is None or old.data_ptr() != ws.data_ptr():
            ws[:64].zero_()      # ws[0] = sticky "a peer CTA never showed up" flag
        return ws

    def lstm_tc_check(self):
        """Raise if a tensor-core recurrence launch gave up waiting for a peer CTA (ws[0] != 0)."""
        for name, t in self.ws.items():
            if name.startswith("lstm_tc_ws_") and int(t[0]) != 0:
                raise MmdaError(f"{name}: a tensor-core recurrence launch timed out waiting for a peer CTA")

    def _launch_gate(self, gate, m, layer, tcws):
        """The text recurrence launches cooperatively (every CTA resident at once): the small
        visual / acoustic recurrences of a layer must not grab SMs just before it.  The text
        stream (enqueued first) marks the point where it reaches its own launch of that layer in
        ``gate``; the side streams wait for that point, so the launches become eligible together
        and stream priority puts the text CTAs first."""
        if m == "t":
            if tcws is not None:
                gate[layer] = self.k.mark()
        else:
            self.k.wait(gate.get(layer))

    # ---------------------------------------------------------------- forward --------------
    def _encode(self, m, X, pk, train, P, gate):
        """reference src/models.py:163-180 + :203 for modality m on the packed rows X (N,I);
        ``gate``: the launch points shared with the other modalities (`_launch_gate`)."""
        k, H = self.k, self.H[m]
        r1, r2, ln = ENC[m]
        N, B, Tmax = pk["N"], pk["B"], pk["Tmax"]
        utt = self.buf(f"utt_{m}", B, 4 * H)
        G1 = self.buf(f"G1_{m}", N, 8 * H)
        Y1 = self.buf(f"Y1_{m}", N, 2 * H)
        C1 = self.buf(f"C1_{m}", N, 2 * H)
        Y1n = self.pbuf(f"Y1n_{m}", N, 2 * H)
        G2 = self.buf(f"G2_{m}", N, 8 * H)
        Y2 = self.buf(f"Y2_{m}", N, 2 * H)
        C2 = self.buf(f"C2_{m}", N, 2 * H)
        mu = self.buf(f"ln_mu_{m}", N)
        rs = self.buf(f"ln_rs_{m}", N)
        if self.gru:
            P = {**P, **self._gru_overlay(m, P, "expand")}
        for G, Xin, r in ((G1, X, r1), (G2, Y1n, r2)):
            if r == r2:
                k.layernorm(Y1, None, P[f"{ln}.weight"], P[f"{ln}.bias"], Y1n, mu, rs)
            I = Xin.shape[1]
            # both directions in ONE GEMM against the stacked, gate-interleaved weight copy:
            # G[N][2][H][4] = Xin * Wst^T + (b_ih + b_hh), 3xTF32 in either precision mode
            Wst, bst = self._pack_weights(r, P, H, I)
            Xp = self._prep(f"tcX_{r}", Xin, kind=0)
            k.gemm_tc(0, 0, 0, N, 8 * H, I, Xp, Wst, G, bias=bst)
            Y, C = (Y1, C1) if r == r1 else (Y2, C2)
            o_f, o_r = (0, 2 * H) if r == r1 else (H, 3 * H)
            if self.gru:
                k._c("mmda_gru_forward", _ptr(G), _ptr(P[f"{r}.weight_hh_l0"]),
                     _ptr(P[f"{r}.weight_hh_l0_reverse"]), _ptr(Y), _ptr(pk["lens"]),
                     _ptr(pk["sidx"]), _ptr(pk["off"]), _ptr(utt), 4 * H, o_f, o_r, B, H, Tmax,
                     int(train))
                continue
            tcws = self._lstm_tc_ws(m, B, H, Tmax)
            if r == r1:
                self._launch_gate(gate, m, 1, tcws)
            if tcws is not None:
                k._c("mmda_lstm_tc_forward", _ptr(G), _ptr(P[f"{r}.weight_hh_l0"]),
                     _ptr(P[f"{r}.weight_hh_l0_reverse"]), _ptr(Y), _ptr(C), _ptr(pk["lens"]),
                     _ptr(pk["sidx"]), _ptr(pk["off"]), _ptr(utt), 4 * H, o_f, o_r, B, H, Tmax,
                     int(train), _ptr(tcws))
            else:
                k._c("mmda_lstm_forward", _ptr(G), _ptr(P[f"{r}.weight_hh_l0"]),
                     _ptr(P[f"{r}.weight_hh_l0_reverse"]), _ptr(Y), _ptr(C), _ptr(pk["lens"]),
                     _ptr(pk["sidx"]), _ptr(pk["off"]), _ptr(utt), 4 * H, o_f, o_r, B, H, Tmax,
                     int(train))
        return utt

    def forward(self, sentences, visual, acoustic, lengths, train: bool, want_sp: bool = True,
                dropout: Optional[bool] = None, seed_dev: Optional[torch.Tensor] = None,
                utt_text: Optional[torch.Tensor] = None, after_heads=None):
        """Returns a dict of device tensors (views into the workspace, valid until the next call).
        ``train`` keeps what the backward needs; ``dropout`` (default: = model.training) enables
        the five Bernoulli sites."""
        k, cfg, d, NC = self.k, self.cfg, self.d, self.NC
        P = self.params()
        k.bind_stream()
        k.det = torch.are_deterministic_algorithms_enabled()
        if self.use_bert != (utt_text is not None):
            raise MmdaError("utt_text (masked-mean BERT output) is required iff config.use_bert")
        for name, t in (("sentences", sentences), ("visual", visual), ("acoustic", acoustic)):
            if name == "sentences" and self.use_bert:
                continue
            if not t.is_cuda and not _DRYRUN:
                raise MmdaError(f"{name} must be a CUDA tensor (reference moves it with to_gpu)")
        pk = self._pack(lengths)
        B, N, Tmax = pk["B"], pk["N"], pk["Tmax"]
        if not self.use_bert and (sentences.shape[0] < Tmax or sentences.shape[1] != B):
            raise MmdaError(f"sentences {tuple(sentences.shape)} inconsistent with lengths")
        drop = self.model.training if dropout is None else dropout
        self.drop_on = bool(drop)
        self.step_id += 1
        # dropout seed: host counter, or (graph-replayable) a constant plus the device step counter
        seed = self.seed if seed_dev is not None else \
            (self.seed * 1000003 + self.step_id) & 0xFFFFFFFFFFFFFFFF
        self.cur_seed, self.seed_dev = seed, seed_dev
        p_cls = float(cfg.dropout) if drop else 0.0
        p_att = ATT_P if drop else 0.0
        self.p_cls, self.p_att = p_cls, p_att
        # nn.RReLU draws its slopes where dropout is on and uses the mean slope otherwise: the
        # linear then runs without an epilogue and the RReLU pass follows in place
        self.rrelu_train = bool(drop) and self.act_id == ACT_RRELU
        act_fwd = ACT_NONE if self.rrelu_train else self.act_id

        # ---- encoders on packed rows (three modalities concurrently) ----
        sent = None if self.use_bert else sentences.contiguous()
        V = 0 if self.use_bert else P["embed.weight"].shape[0]
        X, utt = {}, {}
        srcs = {"v": visual.contiguous(), "a": acoustic.contiguous()}
        for m, src in srcs.items():
            if src.dtype != torch.float32 or src.shape[1] != B or src.shape[2] != self.H[m]:
                raise MmdaError(f"{m} input has shape {tuple(src.shape)} / {src.dtype}")
            X[m] = self.pbuf(f"X_{m}", N, self.H[m])
        if not self.use_bert:
            X["t"] = self.buf("X_t", N, self.H["t"])

        def enc_text():
            if self.use_bert:
                utt["t"] = self.buf("utt_t", B, 768)
                k.add(utt["t"], utt_text.detach().to(torch.float32).contiguous())
                return
            k._c("mmda_embedding_forward", _ptr(P["embed.weight"]), _ptr(sent), _ptr(X["t"]),
                 _ptr(pk["row_t"]), _ptr(pk["row_j"]), _ptr(pk["sidx"]), N, B, self.H["t"], V)
            utt["t"] = self._encode("t", X["t"], pk, train, P, gate)

        def enc_side(m):
            def run():
                k._c("mmda_gather_rows", _ptr(srcs[m]), _ptr(X[m]), X[m].stride(0), _ptr(pk["row_t"]),
                     _ptr(pk["row_j"]), _ptr(pk["sidx"]), N, B, self.H[m])
                utt[m] = self._encode(m, X[m], pk, train, P, gate)
            return run

        self.saved = dict(pk=pk, sent=sent, X=X, train=train, srcs=srcs)
        gate = {}
        self._fork({"t": enc_text, "v": enc_side("v"), "a": enc_side("a")},
                   text_first=not self.gru and not self.use_bert)

        # ---- heads: project -> private/shared -> recon (src/models.py:254-279) ----
        A = self.buf("A", 3, B, d)             # activation output (pre-LN)
        O = self.buf("O", 3, B, d)             # utt_m_orig
        X0 = self.buf("X0", B, 6, d)           # tokens [p_t,p_v,p_a,s_t,s_v,s_a]
        SUM = self.buf("SUM", 3, B, d)         # utt_m = private + shared
        R = self.buf("R", 3, B, d)             # utt_m_recon
        pmu = self.buf("proj_mu", 3, B)
        prs = self.buf("proj_rs", 3, B)
        X0f = X0.view(B, 6 * d)
        def head_fwd(i, m):
            def run():
                k.linear(utt[m], P[f"project_{m}.project_{m}.weight"],
                         P[f"project_{m}.project_{m}.bias"], A[i], act=act_fwd)
                if self.rrelu_train:
                    k.rrelu(A[i], seed, SID_RRELU_PROJECT + i, seed_dev)
                k.layernorm(A[i], None, P[f"project_{m}.project_{m}_layer_norm.weight"],
                            P[f"project_{m}.project_{m}_layer_norm.bias"], O[i], pmu[i], prs[i])
                tag = PRIV_TAG[m]
                k.linear(O[i], P[f"private_{m}.private_{m}_{tag}.weight"],
                         P[f"private_{m}.private_{m}_{tag}.bias"], X0f[:, i * d:(i + 1) * d],
                         act=ACT_SIGMOID)
                k.linear(O[i], P["shared.shared_1.weight"], P["shared.shared_1.bias"],
                         X0f[:, (3 + i) * d:(4 + i) * d], act=ACT_SIGMOID)
                k.add(SUM[i], X0f[:, i * d:(i + 1) * d], X0f[:, (3 + i) * d:(4 + i) * d])
                k.linear(SUM[i], P[f"recon_{m}.recon_{m}_1.weight"],
                         P[f"recon_{m}.recon_{m}_1.bias"], R[i])
            return run

        self._fork({m: head_fwd(i, m) for i, m in enumerate(MODS)})
        if after_heads is not None:
            # the six tokens (X0) are complete: the fused trainer forks the token-only part of the
            # losses (DiffLoss / CMD) from here, beside the fusion layer
            after_heads()
        out = {}
        if self.adversarial:
            # models.py:219-227: domain_label_m = discriminator(GradReverse(utt_shared_m)); the
            # reversal only matters in the backward
            DHp = self.buf("DHpre", 3, B, d)      # activation output (pre-dropout)
            DH = self.buf("DH", 3, B, d)
            DL = self.buf("DL", 3, B, 3)
            for i, m in enumerate(MODS):
                k.linear(X0f[:, (3 + i) * d:(4 + i) * d],
                         P["discriminator.discriminator_layer_1.weight"],
                         P["discriminator.discriminator_layer_1.bias"], DHp[i], act=act_fwd)
                if self.rrelu_train:
                    k.rrelu(DHp[i], seed, SID_RRELU_DISC + i, seed_dev)
                if p_cls > 0:
                    k.dropout(DHp[i], DH[i], p_cls, seed, 6 + i, seed_dev)
                else:
                    k.add(DH[i], DHp[i])
                k.linear(DH[i], P["discriminator.discriminator_layer_2.weight"],
                         P["discriminator.discriminator_layer_2.bias"], DL[i])
                out[f"domain_label_{m}"] = DL[i]
            out["domain"] = DL
        if want_sp:        # outputs no loss reads (src/models.py:234-237); kept for the contract
            SP = self.buf("SP", 4, B, 4)
            smean = self.buf("smean", B, d)
            w, b = (P["sp_discriminator.sp_discriminator_layer_1.weight"],
                    P["sp_discriminator.sp_discriminator_layer_1.bias"])
            for i in range(3):
                k.linear(X0f[:, i * d:(i + 1) * d], w, b, SP[i])
            k.add(smean, X0f[:, 3 * d:4 * d], X0f[:, 4 * d:5 * d], 1.0 / 3.0, 1.0 / 3.0)
            k.add(smean, smean, X0f[:, 5 * d:6 * d], 1.0, 1.0 / 3.0)
            k.linear(smean, w, b, SP[3])
            for i, m in enumerate(MODS):
                out[f"shared_or_private_p_{m}"] = SP[i]
            out["shared_or_private_s"] = SP[3]

        # ---- fusion: post-norm encoder layer over the 6 tokens of each sample ----
        rows = B * 6
        Xr = X0.view(rows, d)
        QKV = self.buf("QKV", rows, 3 * d)
        PR = self.buf("PROBS", B, NHEAD, 6, 6)
        CTX = self.buf("CTX", rows, d)
        AO = self.buf("AO", rows, d)
        X1 = self.buf("X1", rows, d)
        F1 = self.buf("F1", rows, P[TL + "linear1.weight"].shape[0])
        F2 = self.buf("F2", rows, d)
        X2 = self.buf("X2", rows, d)
        lnm = self.buf("enc_mu", 2, rows)
        lnr = self.buf("enc_rs", 2, rows)
        k.linear(Xr, P[TL + "self_attn.in_proj_weight"], P[TL + "self_attn.in_proj_bias"], QKV)
        k._c("mmda_attention_forward", _ptr(QKV), _ptr(CTX), _ptr(PR), B, 6, NHEAD, d // NHEAD,
             p_att, seed, _ptr(seed_dev), 1)
        k.linear(CTX, P[TL + "self_attn.out_proj.weight"], P[TL + "self_attn.out_proj.bias"], AO)
        if p_att > 0:
            k.dropout(AO, AO, p_att, seed, 2, seed_dev)
        k.layernorm(Xr, AO, P[TL + "norm1.weight"], P[TL + "norm1.bias"], X1, lnm[0], lnr[0])
        FF = F1.shape[1]
        ffn_tc = self._tc_lin_ok(rows, FF, d)
        if ffn_tc:
            self.tc_linear("ffn1", X1, P[TL + "linear1.weight"], P[TL + "linear1.bias"], F1)
            # ReLU + dropout in one pass
            k._c("mmda_act_dropout_forward", _ptr(F1), F1.numel(), ACT_RELU, p_att, seed,
                 _ptr(seed_dev), 3)
        else:
            k.linear(X1, P[TL + "linear1.weight"], P[TL + "linear1.bias"], F1, act=ACT_RELU)
            if p_att > 0:
                k.dropout(F1, F1, p_att, seed, 3, seed_dev)
        if ffn_tc:
            self.tc_linear("ffn2", F1, P[TL + "linear2.weight"], P[TL + "linear2.bias"], F2)
        else:
            k.linear(F1, P[TL + "linear2.weight"], P[TL + "linear2.bias"], F2)
        if p_att > 0:
            k.dropout(F2, F2, p_att, seed, 4, seed_dev)
        k.layernorm(X1, F2, P[TL + "norm2.weight"], P[TL + "norm2.bias"], X2, lnm[1], lnr[1])

        # ---- confidence / classifier / labels (src/models.py:247-249) ----
        Hf = X2.view(B, 6 * d)
        TCP = self.buf("TCP", B, 6)
        SC = self.buf("SCORES", B, NC)
        LAB = self.buf("LABELS", B, NC)
        def head(w, b, out, act):     # Linear(6d -> num_classes): one warp per row
            if out.shape[1] <= 8:
                k._c("mmda_linear_skinny", _ptr(Hf), Hf.stride(0), _ptr(P[w]), _ptr(P[b]), _ptr(out),
                     out.stride(0), B, out.shape[1], Hf.shape[1], act)
            else:
                k.linear(Hf, P[w], P[b], out, act=act)

        cw, cb = "confidence.confidence_layer_1.weight", "confidence.confidence_layer_1.bias"
        sw, sb = "classifier.classifier_layer.weight", "classifier.classifier_layer.bias"
        sc_act = ACT_NONE if p_cls > 0 else ACT_SIGMOID
        head(cw, cb, TCP, ACT_SIGMOID)
        head(sw, sb, SC, sc_act)
        if p_cls > 0:
            k.dropout(SC, SC, p_cls, seed, 5, seed_dev)
            k.act(SC, ACT_SIGMOID)
        k._c("mmda_threshold", _ptr(SC), _ptr(LAB), SC.numel(), float(cfg.threshold))

        for i, m in enumerate(MODS):
            out[f"utterance_{m}"] = utt[m]
            out[f"utt_{m}_orig"] = O[i]
            out[f"utt_private_{m}"] = X0[:, i, :]
            out[f"utt_shared_{m}"] = X0[:, 3 + i, :]
            out[f"utt_{m}"] = SUM[i]
            out[f"utt_{m}_recon"] = R[i]
        out.update(tcp=TCP, scores=SC, labels=LAB, tokens=X0, orig=O, recon=R, fused=Hf)
        self.saved.update(utt=utt, B=B)
        return out

    # ---------------------------------------------------------------- backward -------------
    def backward(self, G: Dict[str, torch.Tensor], d_scores=None, d_tcp=None, d_tokens=None,
                 d_orig=None, d_recon=None, d_sp=None, d_domain=None, on_ready=None):
        """Accumulates parameter gradients into ``G[name]`` (tensors shaped like the parameters).

        d_scores, d_tcp (B,NC); d_tokens (B,6,d) grad wrt [p_t,p_v,p_a,s_t,s_v,s_a]; d_orig,
        d_recon (3,B,d); d_sp (4,B,4); any may be None.  ``on_ready(tag)`` is called after the
        kernels producing the gradients of a parameter group have been enqueued (the
        data-parallel trainer uses it to launch bucketed all-reduces)."""
        k, d, NC = self.k, self.d, self.NC
        P = self.params()
        k.bind_stream()
        k.det = det = torch.are_deterministic_algorithms_enabled()
        sv = self.saved
        if not sv.get("train"):
            raise MmdaError("backward() needs a forward(train=True)")
        B, pk = sv["B"], sv["pk"]
        rows = B * 6
        ws = self.ws
        X0 = self.buf("X0", B, 6, d)
        X0f, Xr = X0.view(B, 6 * d), X0.view(rows, d)
        O, A, SUM = self.buf("O", 3, B, d), self.buf("A", 3, B, d), self.buf("SUM", 3, B, d)
        QKV, PR = self.buf("QKV", rows, 3 * d), self.buf("PROBS", B, NHEAD, 6, 6)
        CTX, AO, X1 = self.buf("CTX", rows, d), self.buf("AO", rows, d), self.buf("X1", rows, d)
        FF = P[TL + "linear1.weight"].shape[0]
        F1, F2, X2 = self.buf("F1", rows, FF), self.buf("F2", rows, d), self.buf("X2", rows, d)
        lnm, lnr = self.buf("enc_mu", 2, rows), self.buf("enc_rs", 2, rows)
        Hf = X2.view(B, 6 * d)
        TCP, SC = self.buf("TCP", B, 6), self.buf("SCORES", B, NC)
        seed, p_att, p_cls, seed_dev = self.cur_seed, self.p_att, self.p_cls, self.seed_dev
        notify = on_ready or (lambda tag: None)
        # weight / bias gradients of the dense layers are leaves of the step's dependency graph:
        # they run on side streams (Kernels.leaf) so that only the dx products sit on the chain
        # to the BPTT launches; joined before a data-parallel all-reduce needs them, else at the end
        k.leaf_on = True
        k._leaf_used = {}

        # ---- classifier / confidence ----
        dHf = self.buf("dHf", B, 6 * d)
        have = False
        if d_scores is not None:
            dl = self.buf("dLOGIT", B, NC)
            k.add(dl, d_scores)
            k.act_bwd(dl, SC, ACT_SIGMOID)
            if p_cls > 0:
                k.dropout(dl, dl, p_cls, seed, 5, seed_dev)
            k.linear_bwd(dl, Hf, P["classifier.classifier_layer.weight"],
                         G["classifier.classifier_layer.weight"],
                         G["classifier.classifier_layer.bias"], dHf, 0.0)
            have = True
        if d_tcp is not None:
            dt = self.buf("dTCPpre", B, 6)
            k.add(dt, d_tcp)
            k.act_bwd(dt, TCP, ACT_SIGMOID)
            k.linear_bwd(dt, Hf, P["confidence.confidence_layer_1.weight"],
                         G["confidence.confidence_layer_1.weight"],
                         G["confidence.confidence_layer_1.bias"], dHf, 1.0 if have else 0.0)
            have = True
        dX0 = self.buf("dX0", B, 6, d)
        dX0f, dXr = dX0.view(B, 6 * d), dX0.view(rows, d)
        if have:
            # ---- fusion layer backward ----
            dS2 = self.buf("dS2", rows, d)
            k.layernorm_bwd(dHf.view(rows, d), X1, F2, P[TL + "norm2.weight"], lnm[1], lnr[1], dS2,
                            G[TL + "norm2.weight"], G[TL + "norm2.bias"])
            dF2 = dS2
            if p_att > 0:
                dF2 = self.buf("dF2", rows, d)
                k.dropout(dS2, dF2, p_att, seed, 4, seed_dev)
            dF1 = self.buf("dF1", rows, FF)
            ffn_tc = self._tc_lin_ok(rows, FF, d)
            if ffn_tc:
                self.tc_linear_bwd("ffn2", dF2, F1, P[TL + "linear2.weight"], G[TL + "linear2.weight"],
                                   G[TL + "linear2.bias"], dF1, False)
            else:
                k.linear_bwd(dF2, F1, P[TL + "linear2.weight"], G[TL + "linear2.weight"],
                             G[TL + "linear2.bias"], dF1, 0.0)
            # dropout' + ReLU' in one pass
            k._c("mmda_dropout_act_backward", _ptr(dF1), _ptr(F1), dF1.numel(), ACT_RELU, p_att,
                 seed, _ptr(seed_dev), 3)
            # dX1 = dS2 + dF1 W1   (accumulate in place into dS2)
            if dF2 is dS2:
                k.join_leaves()      # no dropout: dS2 is still being read as linear2's d(output)
            if ffn_tc:
                self.tc_linear_bwd("ffn1", dF1, X1, P[TL + "linear1.weight"], G[TL + "linear1.weight"],
                                   G[TL + "linear1.bias"], dS2, True)
            else:
                k.linear_bwd(dF1, X1, P[TL + "linear1.weight"], G[TL + "linear1.weight"],
                             G[TL + "linear1.bias"], dS2, 1.0)
            dS1 = self.buf("dS1", rows, d)
            k.layernorm_bwd(dS2, Xr, AO, P[TL + "norm1.weight"], lnm[0], lnr[0], dS1,
                            G[TL + "norm1.weight"], G[TL + "norm1.bias"])
            dAO = dS1
            if p_att > 0:
                dAO = self.buf("dAO", rows, d)
                k.dropout(dS1, dAO, p_att, seed, 2, seed_dev)
            dCTX = self.buf("dCTX", rows, d)
            k.linear_bwd(dAO, CTX, P[TL + "self_attn.out_proj.weight"],
                         G[TL + "self_attn.out_proj.weight"], G[TL + "self_attn.out_proj.bias"],
                         dCTX, 0.0)
            dQKV = self.buf("dQKV", rows, 3 * d)
            k._c("mmda_attention_backward", _ptr(QKV), _ptr(PR), _ptr(dCTX), _ptr(dQKV), B, 6,
                 NHEAD, d // NHEAD, p_att, seed, _ptr(seed_dev), 1)
            # dX0 = dS1 + dQKV W_in
            k.add(dXr, dS1)
            k.linear_bwd(dQKV, Xr, P[TL + "self_attn.in_proj_weight"],
                         G[TL + "self_attn.in_proj_weight"], G[TL + "self_attn.in_proj_bias"],
                         dXr, 1.0)
            if d_tokens is not None:
                k.add(dXr, dXr, d_tokens.view(rows, d))
        elif d_tokens is not None:
            k.add(dXr, d_tokens.view(rows, d))
        else:
            dX0.zero_()
        if on_ready is not None:
            k.join_leaves()
        notify("fusion")

        # ---- adversarial discriminator + gradient reversal (functions.py:9-21) ----
        if d_domain is not None:
            DHp, DH = self.buf("DHpre", 3, B, d), self.buf("DH", 3, B, d)
            w1, w2 = (P["discriminator.discriminator_layer_1.weight"],
                      P["discriminator.discriminator_layer_2.weight"])
            lam = float(self.cfg.reverse_grad_weight)
            for i in range(3):
                dDH = self.buf("dDH", B, d)
                k.linear_bwd(d_domain[i], DH[i], w2, G["discriminator.discriminator_layer_2.weight"],
                             G["discriminator.discriminator_layer_2.bias"], dDH, 0.0)
                if p_cls > 0:
                    k.dropout(dDH, dDH, p_cls, seed, 6 + i, seed_dev)
                self._act_bwd(dDH, DHp[i], SID_RRELU_DISC + i)
                dS = self.buf("dSdom", B, d)
                k.linear_bwd(dDH, X0f[:, (3 + i) * d:(4 + i) * d], w1,
                             G["discriminator.discriminator_layer_1.weight"],
                             G["discriminator.discriminator_layer_1.bias"], dS, 0.0)
                sl = dX0f[:, (3 + i) * d:(4 + i) * d]
                k.add(sl, sl, dS, 1.0, -lam)
                k.join_leaves()      # dDH / dS are reused by the next modality

        # ---- sp discriminator (only if somebody asked for its gradient) ----
        if d_sp is not None:
            w = P["sp_discriminator.sp_discriminator_layer_1.weight"]
            gw, gb = (G["sp_discriminator.sp_discriminator_layer_1.weight"],
                      G["sp_discriminator.sp_discriminator_layer_1.bias"])
            smean = self.buf("smean", B, d)
            dsm = self.buf("dsmean", B, d)
            for i in range(3):
                k.linear_bwd(d_sp[i], X0f[:, i * d:(i + 1) * d], w, gw, gb,
                             dX0f[:, i * d:(i + 1) * d], 1.0)
            k.linear_bwd(d_sp[3], smean, w, gw, gb, dsm, 0.0)
            for i in range(3):
                sl = dX0f[:, (3 + i) * d:(4 + i) * d]
                k.add(sl, sl, dsm, 1.0, 1.0 / 3.0)

        # ---- recon / private / shared / project ----
        dO = self.buf("dO", 3, B, d)
        dA = self.buf("dA", 3, B, d)
        dutt = {m: self.buf(f"dutt_{m}", B, self.utt_dim[m]) for m in MODS}
        pmu, prs = self.buf("proj_mu", 3, B), self.buf("proj_rs", 3, B)
        # the shared encoder's gradient gets a term from each modality's stream: atomically
        # accumulated into one tensor, or (deterministic) one partial per stream, summed below
        sh_part = self.buf("shared_1_part", 3, d * d + d) if det else None

        def head_bwd(i, m):
            def run():
                ps, ss = dX0f[:, i * d:(i + 1) * d], dX0f[:, (3 + i) * d:(4 + i) * d]
                if d_recon is not None:
                    dsum = self.buf(f"dSUM_{m}", B, d)
                    k.linear_bwd(d_recon[i], SUM[i], P[f"recon_{m}.recon_{m}_1.weight"],
                                 G[f"recon_{m}.recon_{m}_1.weight"],
                                 G[f"recon_{m}.recon_{m}_1.bias"], dsum, 0.0)
                    k.add(ps, ps, dsum)
                    k.add(ss, ss, dsum)
                k.act_bwd(ps, X0f[:, i * d:(i + 1) * d], ACT_SIGMOID)
                k.act_bwd(ss, X0f[:, (3 + i) * d:(4 + i) * d], ACT_SIGMOID)
                tag = PRIV_TAG[m]
                has_do = d_orig is not None
                if has_do:
                    k.add(dO[i], d_orig[i])
                k.linear_bwd(ps, O[i], P[f"private_{m}.private_{m}_{tag}.weight"],
                             G[f"private_{m}.private_{m}_{tag}.weight"],
                             G[f"private_{m}.private_{m}_{tag}.bias"], dO[i],
                             1.0 if has_do else 0.0)
                if det:
                    sh_part[i].zero_()
                    k.linear_bwd(ss, O[i], P["shared.shared_1.weight"], sh_part[i, :d * d].view(d, d),
                                 sh_part[i, d * d:], dO[i], 1.0)
                else:
                    k.linear_bwd(ss, O[i], P["shared.shared_1.weight"], G["shared.shared_1.weight"],
                                 G["shared.shared_1.bias"], dO[i], 1.0, dw_split=2)
                k.layernorm_bwd(dO[i], A[i], None, P[f"project_{m}.project_{m}_layer_norm.weight"],
                                pmu[i], prs[i], dA[i],
                                G[f"project_{m}.project_{m}_layer_norm.weight"],
                                G[f"project_{m}.project_{m}_layer_norm.bias"])
                self._act_bwd(dA[i], A[i], SID_RRELU_PROJECT + i)
                k.linear_bwd(dA[i], sv["utt"][m], P[f"project_{m}.project_{m}.weight"],
                             G[f"project_{m}.project_{m}.weight"],
                             G[f"project_{m}.project_{m}.bias"], dutt[m], 0.0)
            return run

        self._fork({m: head_bwd(i, m) for i, m in enumerate(MODS)})
        if det:
            k.join_leaves()
            k._c("mmda_fixed_order_sum", _ptr(sh_part), 3, d * d + d, d * d + d,
                 _ptr(G["shared.shared_1.weight"]), _ptr(G["shared.shared_1.bias"]), d * d)
        if on_ready is not None:
            k.join_leaves()
        notify("heads")

        # ---- encoders: BPTT + hoisted weight-gradient GEMMs ----
        def enc_bwd(m):
            def run():
                if not (m == "t" and self.use_bert):
                    self._encode_backward(m, dutt[m], G, pk, P, notify, gate)
                notify(f"enc_{m}")       # on the stream that produced the gradients
            return run

        # The text BPTT launches cooperatively on ~120 SMs: if the small visual / acoustic BPTT
        # kernels get there first it has to wait for them to drain (0.3 ms, measured).  So the
        # text stream is enqueued first and the side streams hold each BPTT launch until the text
        # stream has reached its own launch point of that layer: the launches become eligible
        # together, the text CTAs are placed first (enqueue order) and the small kernels run on the
        # SMs the text kernel leaves free (measured 4.54 ms/step; waiting for the text launch to
        # complete 4.87, no gate 4.56).  The recurrence kernels clean their exchange flags
        # themselves, so no memset node sits between that point and the launch.
        gate = {}
        self._fork({m: enc_bwd(m) for m in MODS}, text_first=not self.gru)
        k.join_leaves()
        k.leaf_on = False
        return dutt["t"] if self.use_bert else None

    def _act_bwd(self, dy, y, sid):
        """dy *= act'(y) for config.activation; training-mode RReLU redraws the forward's slopes
        of random-number stream sid"""
        if self.rrelu_train:
            self.k.rrelu_bwd(dy, y, self.cur_seed, sid, self.seed_dev)
        else:
            self.k.act_bwd(dy, y, self.act_id)

    def _encode_backward(self, m, dutt, G, pk, P, notify, gate):
        """BPTT of both layers of modality m + the hoisted weight-gradient GEMMs.  The recurrence
        and the dX GEMM form the critical path; the weight-gradient work of a layer (h_prev shift,
        dW_ih, dW_hh, bias column sums) is pushed to side streams so it overlaps the next BPTT
        kernel (which leaves 36 of the 148 SMs free).  ``gate``: as in `_encode`."""
        k, H = self.k, self.H[m]
        r1, r2, ln = ENC[m]
        N, B, Tmax = pk["N"], pk["B"], pk["Tmax"]
        X = self.saved["X"][m]
        G1, G2 = self.buf(f"G1_{m}", N, 8 * H), self.buf(f"G2_{m}", N, 8 * H)
        Y1, Y2 = self.buf(f"Y1_{m}", N, 2 * H), self.buf(f"Y2_{m}", N, 2 * H)
        C1, C2 = self.buf(f"C1_{m}", N, 2 * H), self.buf(f"C2_{m}", N, 2 * H)
        Y1n = self.pbuf(f"Y1n_{m}", N, 2 * H)
        mu, rs = self.buf(f"ln_mu_{m}", N), self.buf(f"ln_rs_{m}", N)
        nbytes = LIB.raw("mmda_lstm_scratch_bytes")(B, H)
        if nbytes < 0:
            raise MmdaError(LIB.raw("mmda_last_error")().decode())
        scratch = self.buf(f"lstm_scratch_{m}", max(1, nbytes // 4))
        dY1n = self.pbuf(f"dY1n_{m}", N, 2 * H)
        dY1 = self.buf(f"dY1_{m}", N, 2 * H)
        wg_roles = []
        G_real = G
        if self.gru:
            P = {**P, **self._gru_overlay(m, P, "weights")}      # expanded by the forward
            G = {**G, **self._gru_overlay(m, P, "grads")}
        for r, Gt, Y, C, Xin, dy, (o_f, o_r) in ((r2, G2, Y2, C2, Y1n, None, (H, 3 * H)),
                                                 (r1, G1, Y1, C1, X, dY1, (0, 2 * H))):
            if r == r1:
                k.layernorm_bwd(dY1n, Y1, None, P[f"{ln}.weight"], mu, rs, dY1, G[f"{ln}.weight"],
                                G[f"{ln}.bias"])
            tcws = self._lstm_tc_ws(m, B, H, Tmax)
            self._launch_gate(gate, m, 2 if r == r2 else 1, tcws)
            if tcws is not None:
                k._c("mmda_lstm_tc_backward", _ptr(Gt), _ptr(P[f"{r}.weight_hh_l0"]),
                     _ptr(P[f"{r}.weight_hh_l0_reverse"]), _ptr(C), _ptr(dy), _ptr(dutt), 4 * H, o_f,
                     o_r, _ptr(pk["lens"]), _ptr(pk["sidx"]), _ptr(pk["off"]), B, H, Tmax,
                     _ptr(tcws))
            else:
                k._c("mmda_gru_backward" if self.gru else "mmda_lstm_backward", _ptr(Gt),
                     _ptr(P[f"{r}.weight_hh_l0"]), _ptr(P[f"{r}.weight_hh_l0_reverse"]),
                     _ptr(Y if self.gru else C), _ptr(dy), _ptr(dutt), 4 * H, o_f,
                     o_r, _ptr(pk["lens"]), _ptr(pk["sidx"]), _ptr(pk["off"]), _ptr(scratch), B, H,
                     Tmax)
            if pk["padded"]:
                # padding rows of d(gates) still hold the forward GEMM's values: zero them before
                # the weight-gradient / dX GEMMs and bias column sums reduce over all N rows
                k._c("mmda_zero_tail_rows", _ptr(Gt), 8 * H, _ptr(pk["n_dev"]), N)
            I = Xin.shape[1]
            # 3xTF32 like the forward: weight / activation gradients are sums with heavy
            # cancellation, where bf16 operands cost several percent (measured 4-13 %)
            dGp = self._prep(f"tcdG_{r}", Gt, kind=0)
            Xp = self._prep(f"tcX_{r}", Xin, kind=0)          # the fp32 tensor itself
            Wst = self._prep_buf(f"tcW_{r}", 8 * H, I, 0, split=True)   # packed by the forward

            def wgrad_dir(di):
                # dG columns are gate-interleaved (u*4+g): c_ilv=H stores row u*4+g at g*H+u
                suf = ("", "_reverse")[di]
                dG = Gt[:, di * 4 * H:(di + 1) * 4 * H]
                # contract over tokens: both operands MN-major, auto split-K
                dGd = self._cols(dGp, di * 4 * H, (di + 1) * 4 * H)
                k.gemm_tc(0, 1, 1, 4 * H, I, N, dGd, Xp, G[f"{r}.weight_ih_l0{suf}"], mode=1,
                          split_k=0, c_ilv=H)
                k.gemm_tc(0, 1, 1, 4 * H, H, N, dGd, HPp[di], G[f"{r}.weight_hh_l0{suf}"], mode=1,
                          split_k=0, c_ilv=H)
                k.colsum(dG, G[f"{r}.bias_ih_l0{suf}"], G[f"{r}.bias_hh_l0{suf}"], ilv=H)
                if self.gru:     # 4-slot gradients -> the (3H, .) parameters' gradients
                    k._c("mmda_gru_fold_grads", *[_ptr(G[f"{r}.{kk}{suf}"]) for kk in self._RNN_KEYS],
                         H, I, *[_ptr(G_real[f"{r}.{kk}{suf}"]) for kk in self._RNN_KEYS])

            # one side stream per (layer, direction): the weight-gradient GEMMs of the second
            # layer must not queue in front of the first layer's (they overlap the next BPTT
            # launch and only get the SMs it leaves free)
            wA, wB = ("wg", m, r, 0), ("wg", m, r, 1)
            with k.side(wA, PRIO_LEAF):
                if self.gru:
                    for suf in ("", "_reverse"):
                        for kk in self._RNN_KEYS:
                            G[f"{r}.{kk}{suf}"].zero_()
                Hp = (H + 3) // 4 * 4                 # direction pitch: both slices 16-byte aligned
                HP = self.buf(f"HP_{r}", N, 2 * Hp)
                k._c("mmda_lstm_shift_h", _ptr(Y), _ptr(HP), _ptr(pk["row_t"]), _ptr(pk["row_j"]),
                     _ptr(pk["lens"]), _ptr(pk["off"]), N, H, Hp)
                HPp = [self._prep(f"tcHP_{r}_{di}", HP[:, di * Hp:di * Hp + H], kind=0)
                       for di in (0, 1)]
                common = k.mark()
                wgrad_dir(0)
            with k.side(wB, PRIO_LEAF, after=(common,)):
                wgrad_dir(1)
                if m == "t" and r == r2:
                    # rnn2's gradients are complete once both directions' streams are: let the
                    # data-parallel trainer reduce them under the layer-1 BPTT
                    k.wait(k.mark(wA))
                    notify("enc_t_l2")
            wg_roles += [wA, wB]
            if r == r2 or m == "t":
                dX = dY1n if r == r2 else self.buf("dX_t", N, H)
                # dX = dG [N x 8H] * [W_ih ; W_ih_reverse] (stored [8H][I]: MN-major B)
                k.gemm_tc(0, 0, 1, N, I, 8 * H, dGp, Wst, dX)
                if r == r1:
                    V = P["embed.weight"].shape[0]
                    if k.det:
                        ws = k.det_ws("mmda_embedding_backward_det_workspace_bytes", N, V)
                        k._c("mmda_embedding_backward_det", _ptr(G["embed.weight"]),
                             _ptr(self.saved["sent"]), _ptr(dX), _ptr(pk["row_t"]),
                             _ptr(pk["row_j"]), _ptr(pk["sidx"]), N, B, H, V, _ptr(ws))
                    else:
                        k._c("mmda_embedding_backward", _ptr(G["embed.weight"]),
                             _ptr(self.saved["sent"]), _ptr(dX), _ptr(pk["row_t"]),
                             _ptr(pk["row_j"]), _ptr(pk["sidx"]), N, B, H, V)
                    # the dense embedding gradient (the largest bucket) is complete here, a
                    # millisecond of weight-gradient GEMMs before the rest of the encoder: its
                    # all-reduce runs under them
                    notify("embed")
        k.wait(*[k.mark(role) for role in wg_roles])


# ------------------------------------------------------------------------------------------
# level 1: autograd bridge used by MISA.forward
# ------------------------------------------------------------------------------------------
_DIFF_OUT = ("scores", "tcp") + tuple(f"utt_private_{m}" for m in MODS) + \
    tuple(f"utt_shared_{m}" for m in MODS) + tuple(f"utt_{m}_orig" for m in MODS) + \
    tuple(f"utt_{m}_recon" for m in MODS) + tuple(f"utt_{m}" for m in MODS) + \
    tuple(f"shared_or_private_p_{m}" for m in MODS) + ("shared_or_private_s",)


class _MisaFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, sentences, visual, acoustic, lengths, names, utt_text, *params):
        eng = model.engine
        out = eng.forward(sentences, visual, acoustic, lengths, train=True, want_sp=True,
                          utt_text=utt_text)
        ctx.model, ctx.names, ctx.fwd_step = model, names, eng.step_id
        ctx.set_materialize_grads(False)      # unused outputs arrive as None, not zeros
        res = tuple(out[n].clone() for n in eng.diff_out) + (out["labels"].clone(),)
        ctx.mark_non_differentiable(res[-1])
        return res

    @staticmethod
    def backward(ctx, *g):
        model, eng = ctx.model, ctx.model.engine
        if eng.step_id != ctx.fwd_step:
            raise MmdaError("backward() after a newer forward(): the engine keeps one step of "
                            "saved activations")
        gd = dict(zip(eng.diff_out, g[:-1]))
        dev, d = eng.device, eng.d
        B = eng.saved["B"]

        def stack(keys, shape):
            if all(gd[kk] is None for kk in keys):
                return None
            t = torch.zeros(shape, dtype=torch.float32, device=dev)
            for i, kk in enumerate(keys):
                if gd[kk] is not None:
                    t[i].copy_(gd[kk])
            return t

        d_tok = stack([f"utt_private_{m}" for m in MODS] + [f"utt_shared_{m}" for m in MODS],
                      (6, B, d))
        # utt_m = private + shared feeds both tokens
        for i, m in enumerate(MODS):
            if gd[f"utt_{m}"] is not None:
                if d_tok is None:
                    d_tok = torch.zeros(6, B, d, dtype=torch.float32, device=dev)
                d_tok[i] += gd[f"utt_{m}"]
                d_tok[3 + i] += gd[f"utt_{m}"]
        if d_tok is not None:
            d_tok = d_tok.permute(1, 0, 2).contiguous()
        d_orig = stack([f"utt_{m}_orig" for m in MODS], (3, B, d))
        d_recon = stack([f"utt_{m}_recon" for m in MODS], (3, B, d))
        d_sp = stack([f"shared_or_private_p_{m}" for m in MODS] + ["shared_or_private_s"],
                     (4, B, 4))
        ds = None if gd["scores"] is None else gd["scores"].contiguous()
        dt = None if gd["tcp"] is None else gd["tcp"].contiguous()
        P = eng.params()
        sizes = [P[n].numel() for n in ctx.names]
        arena = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
        G, off = {}, 0
        for n, sz in zip(ctx.names, sizes):
            G[n] = arena[off:off + sz].view(P[n].shape)
            off += sz
        d_dom = stack([f"domain_label_{m}" for m in MODS], (3, B, 3)) if eng.adversarial else None
        d_utt = eng.backward(G, d_scores=ds, d_tcp=dt, d_tokens=d_tok, d_orig=d_orig,
                             d_recon=d_recon, d_sp=d_sp, d_domain=d_dom)
        if d_utt is not None:
            d_utt = d_utt.clone()
        untouched = set()
        if d_sp is None:
            untouched.add("sp_discriminator.")
        if dt is None:
            untouched.add("confidence.")
        if eng.use_bert:
            untouched.add("tlayer_norm.")     # exists in the module but no text LSTM runs
        if eng.adversarial and d_dom is None:
            untouched.add("discriminator.")
        grads = tuple(None if any(n.startswith(u) for u in untouched) else G[n] for n in ctx.names)
        return (None,) * 6 + (d_utt,) + grads


class _BertFunction(torch.autograd.Function):
    """reference src/models.py:186-198 (BertModel -> masked mean over tokens) on the hand-written
    kernels (mmda_b200/bert.py), as one autograd node over the BERT parameters."""

    @staticmethod
    def forward(ctx, model, bert_sent, bert_sent_type, bert_sent_mask, names, *params):
        eng = model.engine
        be = eng.bert
        be.calls = getattr(be, "calls", 0) + 1
        seed = (eng.seed * 7919 + be.calls) & 0xFFFFFFFFFFFFFFFF
        utt = be.forward(bert_sent, bert_sent_type, bert_sent_mask, train=True,
                         drop=model.training, seed=seed)
        ctx.model, ctx.names, ctx.call = model, names, be.calls
        return utt.clone()

    @staticmethod
    def backward(ctx, g):
        be = ctx.model.engine.bert
        if be.calls != ctx.call:
            raise MmdaError("backward() after a newer forward(): the engine keeps one step of "
                            "saved activations")
        P = be.params()
        train = be.trainable()
        G = {n: torch.zeros_like(P[n]) for n in ctx.names if n in train}
        be.backward(G, g.contiguous())
        return (None,) * 5 + tuple(G.get(n) for n in ctx.names)


def misa_apply(model, sentences, visual, acoustic, lengths, bert_sent, bert_sent_type,
               bert_sent_mask):
    eng = model.engine
    named = [(n, p) for n, p in model.named_parameters() if not n.startswith("bertmodel.")]
    utt_text = None
    if eng.use_bert:
        if bert_sent is None:
            raise MmdaError("use_bert=True needs bert_sent / bert_sent_type / bert_sent_mask")
        bnamed = [("bertmodel." + n, p) for n, p in model.bertmodel.named_parameters()]
        if torch.is_grad_enabled() and any(p.requires_grad for _, p in bnamed):
            utt_text = _BertFunction.apply(model, bert_sent, bert_sent_type, bert_sent_mask,
                                           tuple(n for n, _ in bnamed), *[p for _, p in bnamed])
        else:
            utt_text = eng.bert.forward(bert_sent, bert_sent_type, bert_sent_mask, train=False,
                                        drop=False, seed=0).clone()
    needs_grad = torch.is_grad_enabled() and (any(p.requires_grad for _, p in named) or
                                              (utt_text is not None and utt_text.requires_grad))
    if needs_grad:
        names = tuple(n for n, _ in named)
        res = _MisaFunction.apply(model, sentences, visual, acoustic, lengths, names, utt_text,
                                  *[p for _, p in named])
        out = dict(zip(eng.diff_out, res[:-1]))
        out["labels"] = res[-1]
        return out
    o = eng.forward(sentences, visual, acoustic, lengths, train=False, want_sp=True,
                    utt_text=utt_text)
    out = {n: o[n].clone() for n in eng.diff_out}
    out["labels"] = o["labels"].clone()
    return out
