"""BERT-base text encoder on the hand-written kernels (SURVEY.md section 8f row N1).

Replaces ``self.bertmodel(input_ids, attention_mask, token_type_ids)[0]`` + the masked mean at
reference src/models.py:41-45,186-198.  ``model.bertmodel`` stays an HF ``BertModel`` *parameter
container* (same ``state_dict`` keys, so bert-base checkpoints load); none of its ``forward``
methods runs.  Dense layers go through the tcgen05 GEMM (3xTF32 in fp32 mode, bf16 operands in
bf16 mode), everything else through ``csrc/bert.cu`` / ``csrc/elementwise.cu``.

Freeze contract (src/solver.py:66-73): parameters with ``requires_grad=False`` get no weight
gradient; the data gradient still flows through every layer down to the lowest trainable tensor
(the embeddings stay trainable in the reference, so all 12 layers run their dgrad).  The pooler
is never used: its gradients stay ``None``.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from ._lib import LIB, MmdaError

PFX = "bertmodel."


def _ptr(t):
    return None if t is None else t.data_ptr()


class BertEngine:
    def __init__(self, eng):
        self.eng, self.k = eng, eng.k
        bc = eng.model.bertmodel.config
        self.H, self.nh, self.I, self.L = (bc.hidden_size, bc.num_attention_heads,
                                           bc.intermediate_size, bc.num_hidden_layers)
        self.eps = float(bc.layer_norm_eps)
        self.p_h, self.p_a = float(bc.hidden_dropout_prob), float(bc.attention_probs_dropout_prob)
        self.V, self.max_pos = bc.vocab_size, bc.max_position_embeddings
        if bc.hidden_act != "gelu":
            raise MmdaError(f"bert: hidden_act={bc.hidden_act!r} (erf GELU only)")
        if getattr(bc, "position_embedding_type", "absolute") != "absolute":
            raise MmdaError("bert: absolute position embeddings only")
        if self.H != self.nh * 64:
            raise MmdaError("bert: head_dim must be 64 (bert-base geometry)")
        self._pver = None
        self.saved = None
        self._wcache, self._par = {}, {}
        self._resident_max = {}

    # ------------------------------------------------------------------ parameters ---------
    def params(self) -> Dict[str, torch.Tensor]:
        ps = list(self.eng.model.bertmodel.named_parameters())
        ver = tuple(p.data_ptr() for _, p in ps)
        if ver != self._pver:
            from . import engine as _engine
            for n, p in ps:
                if _engine._DRYRUN:
                    continue
                if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous()):
                    raise MmdaError(f"bert parameter {n} must be a contiguous CUDA float32 tensor "
                                    "(no CPU fallback)")
            self._P = {PFX + n: p.data for n, p in ps}
            self._par = {PFX + n: p for n, p in ps}
            self._wcache = {}
            self._pver = ver
        return self._P

    def trainable(self):
        return {PFX + n for n, p in self.eng.model.bertmodel.named_parameters()
                if p.requires_grad and not n.startswith("pooler.")}

    # ------------------------------------------------------------------ GEMM helpers -------
    def _op(self, name, x):
        """tensor-core operand copy (hi/lo tf32 split or bf16) of the 2-D fp32 view x"""
        return self.eng._prep(name, x)

    def _wop(self, P, name):
        """Tensor-core operand copy of a weight: made once per step for trainable weights, once per
        (tensor version, storage) for frozen ones (layers 0-8 under Solver.build's freeze,
        solver.py:69-73) -- their copies live in per-weight workspace buffers nobody else writes.
        In-place edits through ``param.data`` do not bump the version: call ``drop_weight_cache()``
        after such an edit."""
        ops = self._wops
        if name not in ops:
            par = self._par.get(name)
            if par is not None and not par.requires_grad:
                ver = (par._version, par.data_ptr(), self.eng.tc_kind)
                ent = self._wcache.get(name)
                if ent is None or ent[0] != ver:
                    ent = (ver, self.eng._prep("bertW_" + name, P[name], split=True))
                    self._wcache[name] = ent
                ops[name] = ent[1]
            else:
                ops[name] = self.eng._prep("bertW_" + name, P[name], split=True)
        return ops[name]

    def _wqkv(self, P, l):
        """bf16 mode: the stacked [Wq; Wk; Wv] operand copy ([3H][H]) and bias ([3H]) of layer l,
        cached like `_wop` (per step if any of the six tensors trains, else per version)."""
        key = f"qkv{l}"
        if key in self._wops:
            return self._wops[key]
        H, eng = self.H, self.eng
        Lp = f"{PFX}encoder.layer.{l}.attention.self."
        names = [Lp + f"{nm}.{wb}" for nm in ("query", "key", "value") for wb in ("weight", "bias")]
        pars = [self._par[n] for n in names]
        frozen = not any(p.requires_grad for p in pars)
        ver = tuple((p._version, p.data_ptr()) for p in pars)
        ent = self._wcache.get(key) if frozen else None
        if ent is None or ent[0] != ver:
            W = eng._prep_buf(f"bertWqkv_{l}", 3 * H, H, 1)
            b = eng.buf(f"bert_bqkv_{l}", 3 * H)
            for j in range(3):
                eng._prep(f"bertWqkv_{l}", P[names[2 * j]], out=W, row0=j * H, kind=1)
                b[j * H:(j + 1) * H].copy_(P[names[2 * j + 1]], non_blocking=True)
            ent = (ver, (W, b))
            if frozen:
                self._wcache[key] = ent
        self._wops[key] = ent[1]
        return ent[1]

    def drop_weight_cache(self):
        self._wcache = {}

    def _mm(self, a_mn, b_mn, M, N, K, A, B, C, bias=None, acc=False):
        self.k.gemm_tc(self.eng.tc_kind, a_mn, b_mn, M, N, K, A, B, C, bias=bias,
                       mode=1 if acc else 0, split_k=0 if acc else 1)

    def _gelu(self, l, pre, M):
        """GELU of layer l's intermediate pre-activation -> tensor-core operand.  In bf16 mode the
        activation only ever feeds tcgen05 GEMMs, so the kernel writes the bf16 copy directly."""
        I = self.I
        if self.eng.tc_kind == 1:
            act_bf = self.eng.buf(f"bert_actbf_{l}", M, I, dtype=torch.bfloat16)
            self.k._c("mmda_gelu_forward", _ptr(pre), None, _ptr(act_bf), M * I)
            return act_bf, None
        act = self.eng.buf(f"bert_act_{l}", M, I)
        self.k._c("mmda_gelu_forward", _ptr(pre), _ptr(act), None, M * I)
        return self._op("bert_opI", act)

    def _att_sfx(self, S, train):
        """Entry-point suffix of the attention core at sequence length S.  bf16 mode runs it on the
        tensor pipe up to 64 tokens; the shared-memory resident fp32 kernels take what fits them
        (S <= 84 with a backward, S <= 116 without); longer sequences go to the tiled kernels
        (`_tiled_mma` in bf16 mode, `_tiled` in fp32 mode), which hold no S x S buffer."""
        bf = self.eng.tc_kind == 1
        if bf and S <= 64:
            return "_mma"
        key = 1 if train else 0
        if key not in self._resident_max:
            self._resident_max[key] = int(LIB.raw("mmda_bert_attention_resident_max_seq")(key))
        if S <= self._resident_max[key]:
            return ""
        return "_tiled_mma" if bf else "_tiled"

    def _opbuf(self, name, M):
        """bf16 operand buffer a producer kernel writes directly (bf16 mode), else None"""
        return self.eng._prep_buf(name, M, self.H, 1)[0] if self.eng.tc_kind == 1 else None

    def _drop_ln(self, x, res, g, b, y, y_bf, mean, rstd, p, seed, seed_dev, stream_id):
        """y = LN(dropout(x) + res); x := dropout(x); optional bf16 operand copy of y"""
        self.k._c("mmda_dropout_layernorm_forward", _ptr(x), x.stride(0), _ptr(res), res.stride(0),
                  _ptr(g), _ptr(b), _ptr(y), y.stride(0), _ptr(y_bf), _ptr(mean), _ptr(rstd),
                  x.shape[0], x.shape[1], self.eps, p, seed, _ptr(seed_dev), stream_id)

    def _ln_bwd_drop(self, dy, x, res, g, mean, rstd, dx, dg, db, ddrop, ddrop_bf, p, seed, seed_dev,
                     stream_id):
        if self.k.det:
            ws = self.k.det_ws("mmda_layernorm_backward_det_workspace_bytes", x.shape[0], x.shape[1])
            self.k._c("mmda_layernorm_backward_dropout_det", _ptr(dy), dy.stride(0), _ptr(x),
                      x.stride(0), _ptr(res), res.stride(0), _ptr(g), _ptr(mean), _ptr(rstd), _ptr(dx),
                      dx.stride(0), _ptr(dg), _ptr(db), x.shape[0], x.shape[1], _ptr(ddrop),
                      _ptr(ddrop_bf), p, seed, _ptr(seed_dev), stream_id, _ptr(ws))
            return
        self.k._c("mmda_layernorm_backward_dropout", _ptr(dy), dy.stride(0), _ptr(x), x.stride(0),
                  _ptr(res), res.stride(0), _ptr(g), _ptr(mean), _ptr(rstd), _ptr(dx), dx.stride(0),
                  _ptr(dg), _ptr(db), x.shape[0], x.shape[1], _ptr(ddrop), _ptr(ddrop_bf), p, seed,
                  _ptr(seed_dev), stream_id)

    def _ln(self, x, res, g, b, y, mean, rstd):
        self.k._c("mmda_layernorm_forward", _ptr(x), x.stride(0), _ptr(res),
                  0 if res is None else res.stride(0), _ptr(g), _ptr(b), _ptr(y), y.stride(0),
                  _ptr(mean), _ptr(rstd), x.shape[0], x.shape[1], self.eps)

    # ------------------------------------------------------------------ forward ------------
    def forward(self, ids, types, mask, train: bool, drop: bool, seed: int,
                seed_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
        """(B,S) int64 ids / token types / attention mask -> utterance_text (B, hidden)."""
        eng, k, H, I, nh = self.eng, self.k, self.H, self.I, self.nh
        eng.params()                 # binds the workspace to the model's device
        P = self.params()
        k.bind_stream()
        if ids.dim() != 2 or ids.shape != mask.shape or ids.shape != types.shape:
            raise MmdaError("bert: bert_sent / bert_sent_type / bert_sent_mask must be (B, S)")
        from . import engine as _engine
        for t in (ids, types, mask):
            if t.dtype != torch.int64 or not (t.is_cuda or _engine._DRYRUN):
                raise MmdaError("bert: inputs must be CUDA int64 tensors")
        ids, types, mask = ids.contiguous(), types.contiguous(), mask.contiguous()
        B, S = ids.shape
        M = B * S
        p_h = self.p_h if drop else 0.0
        p_a = self.p_a if drop else 0.0
        self._wops = {}
        buf = eng.buf
        E = PFX + "embeddings."
        emb = buf("bert_emb", M, H)
        k._c("mmda_bert_embed_forward", _ptr(P[E + "word_embeddings.weight"]),
             _ptr(P[E + "position_embeddings.weight"]), _ptr(P[E + "token_type_embeddings.weight"]),
             _ptr(ids), _ptr(types), B, S, H, self.V, self.max_pos, _ptr(emb))
        stats = buf("bert_ln_stats", 2 * self.L + 1, 2, M)
        x = buf("bert_x_0", M, H)
        self._ln(emb, None, P[E + "LayerNorm.weight"], P[E + "LayerNorm.bias"], x, stats[0, 0],
                 stats[0, 1])
        if p_h > 0:
            k.dropout(x, x, p_h, seed, 200, seed_dev)
        bf = eng.tc_kind == 1
        xop = None                   # bf16 operand copy of x written by the producing kernel
        for l in range(self.L):
            Lp = f"{PFX}encoder.layer.{l}."
            QKV = buf(f"bert_qkv_{l}", M, 3 * H)
            if xop is None:
                xop = self._op("bert_opH", x)
            if bf:       # one N = 3H GEMM against the stacked [Wq; Wk; Wv] operand copy
                Wqkv, bqkv = self._wqkv(P, l)
                self._mm(0, 0, M, 3 * H, H, xop, Wqkv, QKV, bias=bqkv)
            else:
                for j, nm in enumerate(("query", "key", "value")):
                    self._mm(0, 0, M, H, H, xop, self._wop(P, Lp + f"attention.self.{nm}.weight"),
                             QKV[:, j * H:(j + 1) * H], bias=P[Lp + f"attention.self.{nm}.bias"])
            ctx = buf(f"bert_ctx_{l}", M, H)
            sfx = self._att_sfx(S, train)
            if sfx.startswith("_tiled"):     # O(S) per (sample, head): one lse per row, no probs
                lse = buf(f"bert_lse_{l}", B, nh, S) if train else None
                if sfx == "_tiled_mma":
                    ctx_bf = self._opbuf("bert_opH", M)
                    k._c("mmda_bert_attention_forward_tiled_mma", _ptr(QKV), _ptr(mask),
                         _ptr(ctx) if train else None, _ptr(ctx_bf), _ptr(lse), B, S, nh, 64, p_a,
                         seed, _ptr(seed_dev), 201 + 4 * l)
                    ctx_op = (ctx_bf, None)
                else:
                    k._c("mmda_bert_attention_forward_tiled", _ptr(QKV), _ptr(mask), _ptr(ctx),
                         _ptr(lse), B, S, nh, 64, p_a, seed, _ptr(seed_dev), 201 + 4 * l)
                    ctx_op = self._op("bert_opH", ctx)
                probs = None
            else:
                probs = buf(f"bert_probs_{l}", B, nh, S, S) if train else None
            if sfx == "_mma":      # tensor-pipe core: writes the out-projection's bf16 operand itself
                ctx_bf = self._opbuf("bert_opH", M)
                k._c("mmda_bert_attention_forward_mma", _ptr(QKV), _ptr(mask), _ptr(ctx) if train else None,
                     _ptr(ctx_bf), _ptr(probs), B, S, nh, 64, p_a, seed, _ptr(seed_dev), 201 + 4 * l)
                ctx_op = (ctx_bf, None)
            elif not sfx:
                k._c("mmda_bert_attention_forward", _ptr(QKV), _ptr(mask), _ptr(ctx), _ptr(probs), B, S,
                     nh, 64, p_a, seed, _ptr(seed_dev), 201 + 4 * l)
                ctx_op = self._op("bert_opH", ctx)
            ao = buf(f"bert_ao_{l}", M, H)
            self._mm(0, 0, M, H, H, ctx_op,
                     self._wop(P, Lp + "attention.output.dense.weight"), ao,
                     bias=P[Lp + "attention.output.dense.bias"])
            h1 = buf(f"bert_h1_{l}", M, H)
            h1_bf = self._opbuf("bert_opH", M)
            self._drop_ln(ao, x, P[Lp + "attention.output.LayerNorm.weight"],
                          P[Lp + "attention.output.LayerNorm.bias"], h1, h1_bf, stats[1 + 2 * l, 0],
                          stats[1 + 2 * l, 1], p_h, seed, seed_dev, 202 + 4 * l)
            pre = buf(f"bert_pre_{l}", M, I)
            self._mm(0, 0, M, I, H, (h1_bf, None) if bf else self._op("bert_opH", h1),
                     self._wop(P, Lp + "intermediate.dense.weight"), pre,
                     bias=P[Lp + "intermediate.dense.bias"])
            fo = buf(f"bert_fo_{l}", M, H)
            self._mm(0, 0, M, H, I, self._gelu(l, pre, M),
                     self._wop(P, Lp + "output.dense.weight"), fo, bias=P[Lp + "output.dense.bias"])
            xn = buf(f"bert_x_{l + 1}", M, H)
            xn_bf = self._opbuf("bert_opH", M)
            self._drop_ln(fo, h1, P[Lp + "output.LayerNorm.weight"], P[Lp + "output.LayerNorm.bias"],
                          xn, xn_bf, stats[2 + 2 * l, 0], stats[2 + 2 * l, 1], p_h, seed, seed_dev,
                          203 + 4 * l)
            x = xn
            xop = (xn_bf, None) if bf else None
        utt = buf("bert_utt", B, H)
        k._c("mmda_masked_mean_forward", _ptr(x), _ptr(mask), B, S, H, _ptr(utt))
        self.saved = dict(B=B, S=S, ids=ids, types=types, mask=mask, p_h=p_h, p_a=p_a, seed=seed,
                          seed_dev=seed_dev, train=train)
        return utt

    # ------------------------------------------------------------------ backward -----------
    def backward(self, G: Dict[str, torch.Tensor], d_utt: torch.Tensor):
        """Accumulates (+=) the gradients of the trainable BERT tensors into ``G[name]``."""
        sv = self.saved
        if sv is None or not sv["train"]:
            raise MmdaError("bert.backward needs a preceding forward(train=True)")
        eng, k, H, I, nh = self.eng, self.k, self.H, self.I, self.nh
        P = self.params()
        k.bind_stream()
        k.det = torch.are_deterministic_algorithms_enabled()
        B, S, mask = sv["B"], sv["S"], sv["mask"]
        M = B * S
        p_h, p_a, seed, seed_dev = sv["p_h"], sv["p_a"], sv["seed"], sv["seed_dev"]
        buf = eng.buf
        train = {n for n in self.trainable() if n in G}
        E = PFX + "embeddings."
        emb_train = any(n.startswith(E) for n in train)
        lowest = self.L
        for l in range(self.L):
            if any(n.startswith(f"{PFX}encoder.layer.{l}.") for n in train):
                lowest = l
                break
        if emb_train:
            lowest = -1
        if lowest == self.L:
            return
        stats = buf("bert_ln_stats", 2 * self.L + 1, 2, M)
        scr_g, scr_b = buf("bert_scr_g", H), buf("bert_scr_b", H)

        def gw(name):        # gradient destination of a weight, None if frozen
            return G[name] if name in train else None

        def gw_or(name, scratch):
            return G[name] if name in train else scratch

        def wgrad(dy_op, dy, x_op, wname, bname, N, K):
            """dW[N][K] += dy^T x ; db += colsum(dy)   (dy: [M][N], x: [M][K])"""
            if gw(wname) is not None:
                self._mm(1, 1, N, K, M, dy_op, x_op, G[wname], acc=True)
            if gw(bname) is not None:
                k.colsum(dy, G[bname])

        dx = buf("bert_dxA", M, H)
        k._c("mmda_masked_mean_backward", _ptr(d_utt.contiguous()), _ptr(mask), B, S, H, _ptr(dx))
        other = buf("bert_dxB", M, H)
        for l in range(self.L - 1, max(lowest, 0) - 1, -1):
            Lp = f"{PFX}encoder.layer.{l}."
            x = buf(f"bert_x_{l}", M, H)
            QKV, ctx = buf(f"bert_qkv_{l}", M, 3 * H), buf(f"bert_ctx_{l}", M, H)
            ao, h1 = buf(f"bert_ao_{l}", M, H), buf(f"bert_h1_{l}", M, H)
            pre = buf(f"bert_pre_{l}", M, I)
            bf = eng.tc_kind == 1
            fo = buf(f"bert_fo_{l}", M, H)
            # ---- output LayerNorm(fo + h1) ----
            dsum = other
            # LN backward + the dropout that sat on the dense output + (bf16 mode) the operand
            # copy of the result, one kernel; the fp32 copy only where a bias column sum reads it
            dfo_bf = self._opbuf("bert_opH_d", M)
            need32 = (not bf and p_h > 0) or (bf and gw(Lp + "output.dense.bias") is not None)
            dfo = buf("bert_dH", M, H) if need32 else None
            self._ln_bwd_drop(dx, fo, h1, P[Lp + "output.LayerNorm.weight"], stats[2 + 2 * l, 0],
                              stats[2 + 2 * l, 1], dsum, gw_or(Lp + "output.LayerNorm.weight", scr_g),
                              gw_or(Lp + "output.LayerNorm.bias", scr_b), dfo, dfo_bf, p_h, seed,
                              seed_dev, 203 + 4 * l)
            if not bf and p_h == 0:
                dfo = dsum
            dfo_op = (dfo_bf, None) if bf else self._op("bert_opH_d", dfo)
            # ---- output.dense: act [M][I] -> fo [M][H] ----
            dact = buf("bert_dI", M, I)
            self._mm(0, 1, M, I, H, dfo_op, self._wop(P, Lp + "output.dense.weight"), dact)
            if gw(Lp + "output.dense.weight") is not None:
                act_op = (buf(f"bert_actbf_{l}", M, I, dtype=torch.bfloat16), None) if bf else \
                    self._op("bert_opI", buf(f"bert_act_{l}", M, I))
                wgrad(dfo_op, dfo, act_op, Lp + "output.dense.weight", Lp + "output.dense.bias", H, I)
            if bf:     # d(pre) only feeds GEMMs (+ the bias column sum when that bias is trainable)
                dpre_bf = buf("bert_dIbf", M, I, dtype=torch.bfloat16)
                need32 = gw(Lp + "intermediate.dense.bias") is not None
                k._c("mmda_gelu_backward", _ptr(dact), _ptr(pre), _ptr(dact) if need32 else None,
                     _ptr(dpre_bf), M * I)
                dpre_op = (dpre_bf, None)
            else:
                k._c("mmda_gelu_backward", _ptr(dact), _ptr(pre), _ptr(dact), None, M * I)
                dpre_op = self._op("bert_opI_d", dact)
            # ---- intermediate.dense: h1 [M][H] -> pre [M][I]; dh1 = dsum + dpre W_i ----
            self._mm(0, 1, M, H, I, dpre_op, self._wop(P, Lp + "intermediate.dense.weight"), dsum,
                     acc=True)
            if gw(Lp + "intermediate.dense.weight") is not None:
                wgrad(dpre_op, dact, self._op("bert_opH", h1), Lp + "intermediate.dense.weight",
                      Lp + "intermediate.dense.bias", I, H)
            # ---- attention.output LayerNorm(ao + x) ----
            dsum1 = dx
            dao_bf = self._opbuf("bert_opH_d", M)
            need32 = (not bf and p_h > 0) or (bf and gw(Lp + "attention.output.dense.bias") is not None)
            dao = buf("bert_dH", M, H) if need32 else None
            self._ln_bwd_drop(dsum, ao, x, P[Lp + "attention.output.LayerNorm.weight"],
                              stats[1 + 2 * l, 0], stats[1 + 2 * l, 1], dsum1,
                              gw_or(Lp + "attention.output.LayerNorm.weight", scr_g),
                              gw_or(Lp + "attention.output.LayerNorm.bias", scr_b), dao, dao_bf, p_h,
                              seed, seed_dev, 202 + 4 * l)
            if not bf and p_h == 0:
                dao = dsum1
            dao_op = (dao_bf, None) if bf else self._op("bert_opH_d", dao)
            dctx = buf("bert_dctx", M, H)
            self._mm(0, 1, M, H, H, dao_op, self._wop(P, Lp + "attention.output.dense.weight"), dctx)
            if gw(Lp + "attention.output.dense.weight") is not None:
                wgrad(dao_op, dao, self._op("bert_opH", ctx), Lp + "attention.output.dense.weight",
                      Lp + "attention.output.dense.bias", H, H)
            qkv_names = [Lp + f"attention.self.{nm}.{wb}" for nm in ("query", "key", "value")
                         for wb in ("weight", "bias")]
            sfx = self._att_sfx(S, True)
            mma = sfx.endswith("_mma")
            dQKV = buf("bert_dqkv", M, 3 * H)
            if sfx.startswith("_tiled"):
                lse, delta = buf(f"bert_lse_{l}", B, nh, S), buf("bert_att_delta", B, nh, S)
            else:
                probs = buf(f"bert_probs_{l}", B, nh, S, S)
            if mma:      # tensor-pipe core writes the bf16 operand copy of d(qkv) itself; the fp32
                         # tensor only where a bias column sum reads it
                dq_bf = eng._prep_buf("bert_op3H_d", M, 3 * H, 1)[0]
                need32 = any(n.endswith("bias") and n in train for n in qkv_names)
                if sfx == "_tiled_mma":
                    k._c("mmda_bert_attention_backward_tiled_mma", _ptr(QKV), _ptr(mask), _ptr(ctx),
                         _ptr(lse), _ptr(dctx), _ptr(delta), _ptr(dQKV) if need32 else None,
                         _ptr(dq_bf), B, S, nh, 64, p_a, seed, _ptr(seed_dev), 201 + 4 * l)
                else:
                    k._c("mmda_bert_attention_backward_mma", _ptr(QKV), _ptr(probs), _ptr(dctx),
                         _ptr(dQKV) if need32 else None, _ptr(dq_bf), B, S, nh, 64, p_a, seed,
                         _ptr(seed_dev), 201 + 4 * l)
            elif sfx == "_tiled":
                k._c("mmda_bert_attention_backward_tiled", _ptr(QKV), _ptr(mask), _ptr(ctx), _ptr(lse),
                     _ptr(dctx), _ptr(delta), _ptr(dQKV), B, S, nh, 64, p_a, seed, _ptr(seed_dev),
                     201 + 4 * l)
            else:
                k._c("mmda_bert_attention_backward", _ptr(QKV), _ptr(probs), _ptr(dctx), _ptr(dQKV), B, S,
                     nh, 64, p_a, seed, _ptr(seed_dev), 201 + 4 * l)
            if l > lowest or any(n in train for n in qkv_names):
                dq_op = (dq_bf, None) if mma else self._op("bert_op3H_d", dQKV)
                x_op = None
                if l > lowest and bf:       # dx += d(qkv) [M x 3H] * [Wq; Wk; Wv]: one K = 3H GEMM
                    self._mm(0, 1, M, H, 3 * H, dq_op, self._wqkv(P, l)[0], dsum1, acc=True)
                for j, nm in enumerate(("query", "key", "value")):
                    blk = eng._cols(dq_op, j * H, (j + 1) * H)
                    if l > lowest and not bf:      # the layer below (or the embeddings) needs dx
                        self._mm(0, 1, M, H, H, blk, self._wop(P, Lp + f"attention.self.{nm}.weight"),
                                 dsum1, acc=True)
                    wn, bn = Lp + f"attention.self.{nm}.weight", Lp + f"attention.self.{nm}.bias"
                    if gw(wn) is not None:
                        if x_op is None:
                            x_op = self._op("bert_opH", x)
                        wgrad(blk, dQKV[:, j * H:(j + 1) * H], x_op, wn, bn, H, H)
                    elif gw(bn) is not None:
                        k.colsum(dQKV[:, j * H:(j + 1) * H], G[bn])
            dx, other = dsum1, dsum
        if emb_train:
            if p_h > 0:
                k.dropout(dx, dx, p_h, seed, 200, seed_dev)
            emb = buf("bert_emb", M, H)
            demb = other
            k.layernorm_bwd(dx, emb, None, P[E + "LayerNorm.weight"], stats[0, 0], stats[0, 1], demb,
                            gw_or(E + "LayerNorm.weight", scr_g), gw_or(E + "LayerNorm.bias", scr_b))
            grads = (_ptr(gw(E + "word_embeddings.weight")), _ptr(gw(E + "position_embeddings.weight")),
                     _ptr(gw(E + "token_type_embeddings.weight")))
            if k.det:
                ws = k.det_ws("mmda_bert_embed_backward_det_workspace_bytes", B, S, H, self.V)
                k._c("mmda_bert_embed_backward_det", _ptr(demb), _ptr(sv["ids"]), _ptr(sv["types"]), B,
                     S, H, self.V, *grads, _ptr(ws))
            else:
                k._c("mmda_bert_embed_backward", _ptr(demb), _ptr(sv["ids"]), _ptr(sv["types"]), B, S,
                     H, self.V, *grads)
