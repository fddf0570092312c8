"""Reference pieces for the optimizer tests: the fp64 restatement of clip_grad_value_ +
torch.optim.RMSprop that csrc/adam.cu's rmsprop_clip_kernel implements, and the optimizer the
reference's Solver builds from ``config.optimizer`` (src/solver.py:97-99, src/config.py:24-27).
Both are pinned against torch on CPU in test_optimizer_host.py."""
import numpy as np
import torch


def rmsprop_clip_step(p, g, v, lr, clip=1.0, alpha=0.99, eps=1e-8, grad_scale=1.0):
    """clip_grad_value_(clip) then torch.optim.RMSprop (no momentum, not centered, no weight
    decay); ``grad_scale`` multiplies the gradient before clipping.  eps is added after the
    square root, as torch does."""
    g = np.clip(g * grad_scale, -clip, clip)
    v = alpha * v + (1 - alpha) * g * g
    p = p - lr * g / (np.sqrt(v) + eps)
    return p, v


def reference_optimizer(model, cfg):
    """``config.optimizer(filter(requires_grad, parameters()), lr=config.learning_rate)``: the
    torch.optim class ``cfg.optimizer`` names -- a class, an instance of one, or "Adam" /
    "RMSprop" -- with torch's defaults; Adam when the config has no such field."""
    opt = getattr(cfg, "optimizer", "Adam")
    if isinstance(opt, str):
        cls = {"adam": torch.optim.Adam, "rmsprop": torch.optim.RMSprop}[opt.lower()]
    else:
        cls = opt if isinstance(opt, type) else type(opt)
    return cls([p for p in model.parameters() if p.requires_grad], lr=cfg.learning_rate)
