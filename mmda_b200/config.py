"""Configuration object for the MISA hot path.

The reference builds a ``Config`` from argparse (reference ``src/config.py:71-170``) and the
model / solver read plain attributes off it.  ``MisaConfig`` carries exactly the attributes the
hot path reads (SURVEY.md section 8b, row B1) under the same names and with the same defaults, so
either object can be handed to :class:`mmda_b200.MISA`.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Any, Optional


# activation name -> (kernel epilogue id, torch class name).  ids are shared with csrc/common.cuh
ACTIVATIONS = {
    "none": 0,
    "leakyrelu": 1,
    "sigmoid": 2,
    "relu": 3,
    "tanh": 4,
    "elu": 5,
    "hardshrink": 6,
    "hardtanh": 7,
    "rrelu": 8,
}

# torch's defaults, which is what the kernels compute: the reference constructs
# ``config.activation()`` with no arguments (src/models.py:61-127)
ACTIVATION_DEFAULTS = {
    "elu": dict(alpha=1.0),
    "hardshrink": dict(lambd=0.5),
    "hardtanh": dict(min_val=-1.0, max_val=1.0),
    "rrelu": dict(lower=1.0 / 8, upper=1.0 / 3),
}


def activation_name(act: Any) -> str:
    """Map what the reference stores in ``config.activation`` (an ``nn.Module`` *class*,
    reference ``src/config.py:24-27,78-79``), an instance of one, or a plain string onto a kernel
    epilogue name.  An ELU / Hardshrink / Hardtanh / RReLU instance must carry torch's default
    arguments (``inplace`` is free: it does not change the values)."""
    if isinstance(act, str):
        name = act.lower()
    else:
        cls = act if isinstance(act, type) else type(act)
        name = cls.__name__.lower()
    if name not in ACTIVATIONS or name == "none":
        raise ValueError(
            f"activation {act!r} has no sm_100a epilogue in this build "
            f"(supported: {sorted(k for k in ACTIVATIONS if k != 'none')})")
    if not isinstance(act, (str, type)):
        defaults = ACTIVATION_DEFAULTS.get(name, {})
        bad = {k: getattr(act, k) for k, v in defaults.items() if getattr(act, k, v) != v}
        if bad:
            raise ValueError(f"activation {act!r}: only torch's defaults are implemented "
                             f"({', '.join(f'{k}={v}' for k, v in defaults.items())})")
    return name


# optimizers the fused step implements, with the settings the reference constructs them with
# (``config.optimizer(params, lr=...)``, reference src/solver.py:97-99: torch's defaults)
OPTIMIZERS = {
    "Adam": dict(betas=(0.9, 0.999), eps=1e-8, weight_decay=0, amsgrad=False, maximize=False),
    "RMSprop": dict(alpha=0.99, eps=1e-8, weight_decay=0, momentum=0, centered=False, maximize=False),
}


def optimizer_name(opt: Any) -> str:
    """Map what the reference stores in ``config.optimizer`` (a ``torch.optim`` *class*, reference
    ``src/config.py:24-27,76-77``), an instance of one, or a plain string onto "Adam" or
    "RMSprop".  An instance must use the reference's settings (anything but the learning rate at
    torch's defaults); its learning rate is not read: ``learning_rate`` sets it."""
    if isinstance(opt, str):
        name = {k.lower(): k for k in OPTIMIZERS}.get(opt.lower())
    else:
        cls = opt if isinstance(opt, type) else type(opt)
        name = cls.__name__ if cls.__name__ in OPTIMIZERS else None
    if name is None:
        raise ValueError(f"optimizer {opt!r} has no fused step in this build "
                         f"(supported: {sorted(OPTIMIZERS)})")
    defaults = getattr(opt, "defaults", None)
    if not isinstance(opt, (str, type)) and isinstance(defaults, dict):
        bad = {k: defaults[k] for k, v in OPTIMIZERS[name].items()
               if k in defaults and (tuple(defaults[k]) if k == "betas" else defaults[k]) != v}
        if bad:
            raise ValueError(f"{name} with {bad}: only {name}(params, lr) is implemented "
                             f"({', '.join(f'{k}={v}' for k, v in OPTIMIZERS[name].items())})")
    return name


@dataclass
class MisaConfig:
    # --- model (reference src/models.py:20-47, src/config.py:146-154) ---
    embedding_size: int = 300
    visual_size: int = 35
    acoustic_size: int = 74
    num_classes: int = 6
    hidden_size: int = 128
    dropout: float = 0.1
    activation: Any = "leakyrelu"
    extractor: str = "lstm"
    rnncell: str = "lstm"
    use_bert: bool = False
    use_cmd_sim: bool = True
    reverse_grad_weight: float = 1.0
    threshold: float = 0.35
    vocab_size: int = 20000          # len(config.word2id) in the reference
    word2id: Optional[Any] = None
    pretrained_emb: Optional[Any] = None
    # --- solver (reference src/config.py:134-143, src/solver.py:175-186) ---
    data: str = "mosei"
    use_confidNet: bool = False
    diff_weight: float = 0.3
    sim_weight: float = 0.7
    sp_weight: float = 0.0
    recon_weight: float = 0.7
    conf_weight: float = 0.3
    learning_rate: float = 1e-4
    optimizer: Any = "Adam"          # torch.optim.Adam / RMSprop (class or instance) or its name
    clip: float = 1.0
    batch_size: int = 64
    model: str = "MISA"
    # --- this build only ---
    precision: str = "fp32"          # "fp32" | "bf16" (operands of the hoisted input-projection GEMMs)

    def __post_init__(self):
        if self.word2id is None:
            self.word2id = range(self.vocab_size)
        else:
            self.vocab_size = len(self.word2id)


def mosi_config(**kw) -> MisaConfig:
    """BASELINE.json configs[0]: MOSI-shape (300/47/74), batch 64."""
    d = dict(visual_size=47, acoustic_size=74, batch_size=64, data="mosi")
    d.update(kw)
    return MisaConfig(**d)


def mosei_config(**kw) -> MisaConfig:
    """BASELINE.json configs[1]: MOSEI-shape (300/35/74), batch 256."""
    d = dict(visual_size=35, acoustic_size=74, batch_size=256, data="mosei")
    d.update(kw)
    return MisaConfig(**d)
