"""TEST / BENCH INFRASTRUCTURE -- never imported by the product package (lightly_train_b200/).

Runs the reference's OWN method class (`lightly_train._methods.dinov2.dinov2.DINOv2`, unmodified source) without its
absent third-party packages.  The reference source is taken from the directory named by $LIGHTLY_TRAIN_SRC (the `src`
directory of a lightly-train checkout) or from `baseline/_ref` (a `pip install --no-deps --target baseline/_ref` copy).  Its
dependencies that are NOT in this image -- pytorch_lightning, lightly, omegaconf, albumentations, lightning_utilities,
... -- are replaced by stubs:

  * pytorch_lightning.LightningModule  -> `LightningModuleStub` below: an nn.Module with `trainer`, `log_dict`,
    `clip_gradients` (torch clip_grad_norm_) and nothing else.  The fit loop is `run_step` below, which calls the
    reference's hooks in Lightning's automatic-optimisation order (training_step -> backward -> on_before_optimizer_step
    -> configure_gradient_clipping -> optimizer.step -> scheduler.step -> global_step += 1 -> on_train_batch_end).
  * lightly.utils.scheduler.{cosine_schedule, CosineWarmupScheduler}, lightly.utils.optim.update_param_groups,
    lightly.loss.KoLeoLoss, lightly.transforms.utils.IMAGENET_NORMALIZE -> restated from lightly 1.5.x's published
    definitions (the package itself is absent: THESE FOUR ARE UNPINNED, see DESIGN.md section 4).
  * everything else those packages export -> inert placeholders (only ever used as base classes / annotations by code
    outside the training step).

Everything the training step executes inside `lightly_train` (ViT, heads, losses, masking, optimizer groups, EMA, the
method's own training_step_impl / hooks) is the reference's code.
"""
from __future__ import annotations

import importlib.abc
import importlib.machinery
import math
import os
import sys
import types
from pathlib import Path
from typing import Any, Dict, List, Optional

import torch
from torch import Tensor, nn

ROOT = Path(__file__).resolve().parents[1]
CANDIDATES = [Path(p) for p in (os.environ.get("LIGHTLY_TRAIN_SRC"),) if p] + [ROOT / "baseline" / "_ref"]

_STUB_ROOTS = ("pytorch_lightning", "lightly", "lightning_utilities", "omegaconf", "albumentations", "lightning_fabric",
               "wandb", "mlflow", "tensorboard", "cv2", "pydicom", "timm", "xformers", "rfdetr", "ultralytics", "super_gradients",
               "lightning", "torchmetrics", "pycocotools", "onnx", "onnxruntime", "eomt", "matplotlib", "fsspec", "psutil_stub")


def source_root() -> Optional[Path]:
    for c in CANDIDATES:
        try:
            if (c / "lightly_train" / "_methods" / "dinov2" / "dinov2.py").is_file():
                return c
        except OSError:  # e.g. a directory this user may not read
            pass
    return None


def available() -> bool:
    return source_root() is not None


# ---------------------------------------------------------------------------------------------- stubs
class _Placeholder:
    """Inert stand-in: subclassable, callable as a decorator / constructor, usable in annotations and `|` unions."""

    def __init__(self, *a: Any, **k: Any) -> None:
        pass

    def __init_subclass__(cls, **k: Any) -> None:
        pass

    def __call__(self, *a: Any, **k: Any) -> Any:
        if len(a) == 1 and callable(a[0]) and not k:
            return a[0]
        return self

    def __getattr__(self, name: str) -> Any:
        if name.startswith("__"):
            raise AttributeError(name)
        return _Placeholder()

    def __or__(self, other: Any) -> Any:
        return Any

    __ror__ = __or__

    def __class_getitem__(cls, item: Any) -> Any:
        return cls

    def __bool__(self) -> bool:
        return False


class _PlaceholderMeta(type):
    def __getattr__(cls, name: str) -> Any:
        if name.startswith("__"):
            raise AttributeError(name)
        return _Placeholder()

    def __or__(cls, other: Any) -> Any:
        return Any

    __ror__ = __or__


def _placeholder_class(name: str) -> type:
    return _PlaceholderMeta(name, (_Placeholder,), {})


class _StubModule(types.ModuleType):
    def __getattr__(self, name: str) -> Any:
        if name.startswith("__"):
            raise AttributeError(name)
        if name[:1].isupper():
            v: Any = _placeholder_class(name)
        else:
            v = _Placeholder()
        setattr(self, name, v)
        return v


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, fullname, path=None, target=None):
        if fullname.split(".")[0] in _STUB_ROOTS:
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        return None

    def create_module(self, spec):
        m = _StubModule(spec.name)
        m.__path__ = []  # a package: submodule imports come back to this finder
        return m

    def exec_module(self, module):
        _populate(module)


# ---- the pieces the training step really executes -----------------------------------------------------------------
def cosine_schedule(step: int, max_steps: int, start_value: float, end_value: float, period: Optional[int] = None) -> float:
    """lightly.utils.scheduler.cosine_schedule (lightly 1.5.x), restated."""
    if step < 0:
        raise ValueError(f"Current step number {step} can't be negative")
    if max_steps < 1:
        raise ValueError(f"Total step number {max_steps} must be >= 1")
    if period is None and step > max_steps:
        step = max_steps
    if period is not None:
        return end_value + 0.5 * (start_value - end_value) * (1 + math.cos(2 * math.pi * step / period))
    if max_steps == 1:
        return end_value
    if step == max_steps:
        return end_value
    return end_value + 0.5 * (start_value - end_value) * (1 + math.cos(math.pi * step / (max_steps - 1)))


class CosineWarmupScheduler(torch.optim.lr_scheduler.LambdaLR):
    """lightly.utils.scheduler.CosineWarmupScheduler, restated: linear warm-up (epoch+1)/warmup, then cosine to end_value."""

    def __init__(self, optimizer, warmup_epochs: int, max_epochs: int, last_epoch: int = -1, start_value: float = 1.0,
                 end_value: float = 0.001, period: Optional[int] = None, verbose: bool = False) -> None:
        self.warmup_epochs, self.max_epochs = warmup_epochs, max_epochs
        self.start_value, self.end_value, self.period = start_value, end_value, period
        super().__init__(optimizer=optimizer, lr_lambda=self.scale_lr, last_epoch=last_epoch)

    def scale_lr(self, epoch: int) -> float:
        if self.warmup_epochs > 0 and epoch < self.warmup_epochs:
            return self.start_value * (epoch + 1) / self.warmup_epochs
        if self.period is not None:
            return cosine_schedule(epoch - self.warmup_epochs, 1, self.start_value, self.end_value, self.period)
        return cosine_schedule(epoch - self.warmup_epochs, self.max_epochs - self.warmup_epochs, self.start_value, self.end_value)


def update_param_groups(optimizer, default_update: Optional[dict] = None, updates: Optional[List[dict]] = None) -> None:
    """lightly.utils.optim.update_param_groups, restated: per-name key/value updates of optimizer.param_groups."""
    default_update = default_update or {}
    by_name = {u["name"]: u for u in (updates or [])}
    for group in optimizer.param_groups:
        upd = by_name.get(group.get("name"), default_update)
        for k, v in upd.items():
            if k != "name":
                group[k] = v


class KoLeoLoss(nn.Module):
    """lightly.loss.KoLeoLoss (1.5.x), restated: -mean(log(||x_i - x_nn(i)||_2 + eps)) on L2-normalised rows, nearest
    neighbour by largest dot product with the diagonal excluded."""

    def __init__(self, p: float = 2, eps: float = 1e-8) -> None:
        super().__init__()
        self.p, self.eps = p, eps
        self.pairwise_distance = nn.PairwiseDistance(p=p, eps=eps)

    def forward(self, x: Tensor) -> Tensor:
        x = torch.nn.functional.normalize(x, p=2, dim=-1, eps=self.eps)
        cos_sim = torch.mm(x, x.t())
        cos_sim.fill_diagonal_(-2)
        min_idx = torch.argmax(cos_sim, dim=1)
        min_dist = self.pairwise_distance(x, x[min_idx])
        return -torch.mean(torch.log(min_dist + self.eps))


class _Trainer:
    def __init__(self, max_steps: int) -> None:
        self.global_step = 0
        self.estimated_stepping_batches = max_steps
        self.max_epochs = 1
        self.world_size = 1
        self.is_global_zero = True
        self.train_dataloader = None
        self.loggers: list = []


class LightningModuleStub(nn.Module):
    """What the reference method uses of pytorch_lightning.LightningModule during a step."""

    def __init__(self, *a: Any, **k: Any) -> None:
        super().__init__()
        self._trainer_stub: Optional[_Trainer] = None
        self.logged: Dict[str, Any] = {}

    @property
    def trainer(self) -> _Trainer:
        assert self._trainer_stub is not None, "attach a trainer with ref_full.attach_trainer"
        return self._trainer_stub

    @trainer.setter
    def trainer(self, t: _Trainer) -> None:
        self._trainer_stub = t

    @property
    def global_step(self) -> int:
        return self.trainer.global_step

    @property
    def device(self) -> torch.device:
        return next(self.parameters()).device

    def log_dict(self, d, *a: Any, **k: Any) -> None:
        self.logged.update({kk: (float(v) if isinstance(v, Tensor) else v) for kk, v in d.items()})

    def log(self, name, value, *a: Any, **k: Any) -> None:
        self.logged[name] = float(value) if isinstance(value, Tensor) else value

    def clip_gradients(self, optimizer, gradient_clip_val=None, gradient_clip_algorithm=None) -> None:
        assert gradient_clip_algorithm == "norm"
        params = [p for g in optimizer.param_groups for p in g["params"]]
        torch.nn.utils.clip_grad_norm_(params, gradient_clip_val)

    def on_train_batch_end(self, *a: Any, **k: Any) -> None:
        pass

    def save_hyperparameters(self, *a: Any, **k: Any) -> None:
        pass


def _populate(module: types.ModuleType) -> None:
    n = module.__name__
    if n == "pytorch_lightning":
        module.LightningModule = LightningModuleStub
    elif n == "pytorch_lightning.utilities":
        module.rank_zero_only = lambda fn: fn
    elif n == "lightly.loss":
        module.KoLeoLoss = KoLeoLoss
    elif n == "lightly.utils.optim":
        module.update_param_groups = update_param_groups
    elif n == "lightly.utils.scheduler":
        module.cosine_schedule = cosine_schedule
        module.CosineWarmupScheduler = CosineWarmupScheduler
    elif n == "lightly.transforms.utils":
        module.IMAGENET_NORMALIZE = {"mean": [0.485, 0.456, 0.406], "std": [0.229, 0.224, 0.225]}
    elif n == "lightning_utilities.core.imports":
        class RequirementCache:  # every optional requirement reads as "not installed"
            def __init__(self, *a: Any, **k: Any) -> None:
                pass

            def __bool__(self) -> bool:
                return False

        module.RequirementCache = RequirementCache


_installed = False


def install() -> None:
    """Make `lightly_train.<submodule>` importable (package __init__ skipped: it pulls the CLI / data plane)."""
    global _installed
    if _installed:
        return
    src = source_root()
    if src is None:
        raise RuntimeError("reference source not found (set LIGHTLY_TRAIN_SRC or install a copy into baseline/_ref)")
    os.environ["XFORMERS_DISABLED"] = "1"
    for name in list(sys.modules):
        if name.split(".")[0] in ("lightly_train", "lightning_utilities"):
            del sys.modules[name]
    sys.meta_path.append(_StubFinder())
    pkg = types.ModuleType("lightly_train")
    pkg.__path__ = [str(src / "lightly_train")]
    sys.modules["lightly_train"] = pkg
    _installed = True


# ---------------------------------------------------------------------------------------------- driving the method
def build_dinov2(vit_kwargs: Dict[str, Any], method_overrides: Dict[str, Any], global_batch_size: int, max_steps: int,
                 device: str = "cpu", activation_checkpointing: bool = False):
    """Instantiate the reference DINOv2 method around a reference DinoVisionTransformer(**vit_kwargs)."""
    install()
    from lightly_train._methods.dinov2.dinov2 import DINOv2, DINOv2AdamWViTArgs, DINOv2Args  # type: ignore
    from lightly_train._models.dinov2_vit.dinov2_vit import DINOv2ViTModelWrapper  # type: ignore
    from lightly_train._models.dinov2_vit.dinov2_vit_src.models.vision_transformer import DinoVisionTransformer  # type: ignore
    from lightly_train._models.embedding_model import EmbeddingModel  # type: ignore

    vit = DinoVisionTransformer(**vit_kwargs)
    vit.init_weights()
    wrapper = DINOv2ViTModelWrapper(vit)
    emb = EmbeddingModel(wrapped_model=wrapper)
    margs = DINOv2Args(**method_overrides)
    oargs = DINOv2AdamWViTArgs()
    if margs.weight_decay_start == "auto":
        margs.weight_decay_start = oargs.weight_decay
    m = DINOv2(method_args=margs, optimizer_args=oargs, embedding_model=emb, global_batch_size=global_batch_size,
               num_input_channels=vit_kwargs.get("in_chans", 3))
    m.trainer = _Trainer(max_steps)
    if activation_checkpointing:
        m.student_embedding_model.wrapped_model.set_activation_checkpointing(True)
    m.to(device)
    (opt,), (sched,) = m.configure_optimizers()
    return m, opt, sched["scheduler"]


def run_step(m, opt, sched, batch: Dict[str, Any], autocast_device: Optional[str] = None) -> Tensor:
    """One optimisation step in Lightning's automatic-optimisation hook order."""
    opt.zero_grad(set_to_none=True)
    if autocast_device is not None:
        with torch.autocast(autocast_device, dtype=torch.bfloat16):
            res = m.training_step_impl(batch, 0)
    else:
        res = m.training_step_impl(batch, 0)
    res.loss.backward()
    m.on_before_optimizer_step(opt)
    m.configure_gradient_clipping(opt)
    opt.step()
    sched.step()
    m.trainer.global_step += 1
    m.on_train_batch_end(None, batch, 0)
    m.last_log = dict(res.log_dict or {})
    return res.loss.detach()
