"""Evaluation pass on the device (SURVEY.md section 8f, N2): the reference's ``Solver.eval``
(src/solver.py:311-370: eval mode, no grad, forward, cls loss only, predictions thresholded at
``config.threshold``) with the multi-label metrics of src/utils/eval.py accumulated by a kernel,
so a whole dev/test pass costs ONE device->host read instead of per-batch ``.cpu().numpy()``."""
from __future__ import annotations

from typing import Dict, Iterable

import torch

from .engine import _ptr


def metrics_from_stats(stats, num_classes: int) -> Dict[str, float]:
    """stats: the 4+3*NC vector of mmda_eval_accumulate.  Same definitions as
    ``get_accuracy`` (eval.py:14-31, rounded to 4 decimals) and sklearn's precision / recall / F1
    with zero_division -> 0 (eval.py:33-65)."""
    s = [float(x) for x in stats]
    NC = num_classes
    tp, fp, fn = s[4:4 + NC], s[4 + NC:4 + 2 * NC], s[4 + 2 * NC:4 + 3 * NC]
    div = lambda a, b: a / b if b > 0 else 0.0
    prec = [div(tp[c], tp[c] + fp[c]) for c in range(NC)]
    rec = [div(tp[c], tp[c] + fn[c]) for c in range(NC)]
    f1 = [div(2 * tp[c], 2 * tp[c] + fp[c] + fn[c]) for c in range(NC)]
    sup = [tp[c] + fn[c] for c in range(NC)]
    wsum = lambda v: div(sum(v[c] * sup[c] for c in range(NC)), sum(sup))
    TP, FP, FN = sum(tp), sum(fp), sum(fn)
    return {
        "loss": div(s[2], s[3]), "acc": round(div(s[0], s[1]), 4),
        "f1": sum(f1) / NC, "precision": sum(prec) / NC, "recall": sum(rec) / NC,
        "micro_f1": div(2 * TP, 2 * TP + FP + FN), "micro_precision": div(TP, TP + FP),
        "micro_recall": div(TP, TP + FN),
        "weighted_f1": wsum(f1), "weighted_precision": wsum(prec), "weighted_recall": wsum(rec),
    }


@torch.no_grad()
def evaluate(model, batches: Iterable, device=None) -> Dict[str, float]:
    """batches yield objects with ``sentences, visual, acoustic, lengths, labels`` (host or device
    tensors; ``lengths`` on the CPU), and with ``use_bert=True`` also ``bert_sent,
    bert_sent_type, bert_sent_mask``."""
    was_training = model.training
    model.eval()
    eng = model.engine
    dev = device or next(model.parameters()).device
    NC = eng.NC
    stats = torch.zeros(4 + 3 * NC, dtype=torch.float32, device=dev)
    to = lambda t: t.to(dev, non_blocking=True)
    for b in batches:
        utt_text = None
        if eng.use_bert:     # text branch: the BERT encoder's masked mean, no dropout
            utt_text = eng.bert.forward(to(b.bert_sent), to(b.bert_sent_type), to(b.bert_sent_mask),
                                        train=False, drop=False, seed=0)
        out = eng.forward(to(b.sentences), to(b.visual), to(b.acoustic), b.lengths, train=False,
                          want_sp=False, dropout=False, utt_text=utt_text)
        y = to(b.labels).float().contiguous()
        eng.k._c("mmda_eval_accumulate", _ptr(out["scores"]), _ptr(out["labels"]), _ptr(y),
                 _ptr(stats), y.shape[0], NC)
    model.train(was_training)
    return metrics_from_stats(stats.tolist(), NC)
