"""DINOv2 method on B200 kernels.

Mirror of LT/_methods/dinov2/dinov2.py: `DINOv2Args` / `DINOv2AdamWViTArgs` (:70-164), `DINOv2Head` (:167-174)
and the `DINOv2` method (:176-692) -- teacher/student ViTs + projection heads, DINO / iBOT / KoLeo losses,
layer-wise-decay AdamW with cosine weight decay, last-layer lr freeze, gradient clipping and the EMA teacher
update.  The public surface keeps the reference's names (`training_step_impl`, `on_before_optimizer_step`,
`on_train_batch_end`, `TrainingStepResult`, the `train_loss/*` log keys, parameter/buffer names under
`teacher_embedding_model.*`, `student_embedding_model.*`, `{teacher,student}_head.{dino_head,ibot_head}.*`,
`dino_loss.center`, `ibot_loss.center`).

Execution model (B200-first, not the reference's autograd graph): one training step is an explicit schedule
of sm_100a kernel launches -- teacher forward, student forward (global, local), fused CE forward+backward,
head and ViT backward into a flat gradient arena -- followed by ONE fused sweep doing gradient clipping,
AdamW, the EMA teacher update and the bf16 weight-shadow refresh.  `training_step_impl` therefore returns the
loss with gradients already accumulated in `param.grad` (views of the arena); `loss_for_autograd()` offers a
torch.autograd bridge for trainers that insist on calling `loss.backward()` (INTEGRATION.md).
"""
from __future__ import annotations

import atexit
import math
import os
import weakref
from dataclasses import dataclass, field
from typing import Any, Dict, List, Literal, Optional, Tuple

import torch
import torch.distributed as dist
from torch import Tensor, nn

from ... import ops
from ..._arena import CHUNK, Arena
from ..._models.dinov2_vit import DinoVisionTransformer, vit_param_shapes
from .dinov2_head import DINOv2ProjectionHead, head_param_shapes
from .dinov2_loss import DINOLoss, IBOTPatchLoss, sinkhorn_colterm
from .scheduler import cosine_schedule, cosine_warmup_factor, linear_warmup_schedule
from ..._torch_helpers import update_momentum
from ... import _lib
from .utils import MaskingGenerator, create_collated_masks, param_group_settings

# Sinkhorn-Knopp on several ranks: capture the per-iteration [K] all-reduces into the step's CUDA graph (NCCL kernels are
# capturable; 2 x B200 at cfg3: 36.4 ms against 45.7 ms launched eagerly).  B200_GRAPH_NCCL=0 keeps that step eager.
GRAPH_NCCL = os.environ.get("B200_GRAPH_NCCL", "1") == "1"

# A communicator cannot be torn down while a live CUDA graph holds captured NCCL kernels (destroy_process_group blocks for
# ever): methods that captured collectives are tracked here and their graphs are dropped before the process group goes.
_NCCL_GRAPH_HOLDERS: "weakref.WeakSet[DINOv2]" = weakref.WeakSet()
_teardown_hooked = False


def _release_all_nccl_graphs() -> None:
    for m in list(_NCCL_GRAPH_HOLDERS):
        try:
            if torch.cuda.is_available():
                torch.cuda.synchronize()
            m.release_graphs()
        except Exception:  # interpreter shutdown: nothing left to protect
            pass


def _hook_process_group_teardown() -> None:
    global _teardown_hooked
    if _teardown_hooked:
        return
    _teardown_hooked = True
    original = dist.destroy_process_group

    def destroy_process_group(*args: Any, **kwargs: Any) -> Any:
        _release_all_nccl_graphs()
        return original(*args, **kwargs)

    dist.destroy_process_group = destroy_process_group
    atexit.register(_release_all_nccl_graphs)


# where the backbone backward is cut for the middle all-reduce bucket: blocks >= FRAC * depth go out after graph 2
DDP_SPLIT_FRAC = float(os.environ.get("B200_DDP_SPLIT_FRAC", "0.5"))


def _world_size() -> int:
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


@dataclass
class DINOv2Args:
    """LT/_methods/dinov2/dinov2.py:70-153 (same field names and defaults)."""

    ibot_separate_head: bool = False
    hidden_dim: int = 2048
    dino_bottleneck_dim: int = 256
    ibot_bottleneck_dim: int = 256
    output_dim: int = 65536
    batch_norm: bool = False
    student_freeze_last_layer_steps: int = 1250
    student_freeze_backbone_steps: int = 0
    dino_loss_weight: float = 1.0
    ibot_loss_weight: float = 1.0
    koleo_loss_weight: float = 0.1
    center_method: Literal["softmax", "sinkhorn_knopp"] = "softmax"
    center_momentum: float = 0.9
    momentum_start: float = 0.992
    momentum_end: float = 1.0
    student_temp: float = 0.1
    teacher_temp_start: float = 0.04
    teacher_temp_end: float = 0.07
    teacher_temp_warmup_steps: int = 37500
    mask_ratio_min: float = 0.1
    mask_ratio_max: float = 0.5
    mask_probability: float = 0.5
    min_lr: float = 1.0e-06
    warmup_steps: int = 12500
    layerwise_decay: float = 0.9
    patch_embed_lr_multiplier: float = 0.2
    lr_scale_method: Literal["linear", "sqrt"] = "sqrt"
    reference_batch_size: int = 1024
    weight_decay_start: float | Literal["auto"] = "auto"
    weight_decay_end: float = 0.4
    gradient_clip_val: float = 3.0


@dataclass
class DINOv2AdamWViTArgs:
    """LT/_methods/dinov2/dinov2.py:156-164."""

    lr: float = 0.004
    betas: Tuple[float, float] = (0.9, 0.999)
    eps: float = 1e-8
    weight_decay: float = 0.04


@dataclass
class TrainingStepResult:
    """LT/_methods/method.py:41-44."""

    loss: Tensor
    log_dict: Dict[str, Any] = field(default_factory=dict)


class _TrainerState:
    """The three Trainer attributes the reference method reads (tests mock exactly these, test_dinov2.py:54-59)."""

    def __init__(self, max_steps: int) -> None:
        self.global_step = 0
        self.estimated_stepping_batches = max_steps
        self.max_epochs = 1


class DINOv2Head(nn.Module):
    def __init__(self, dino_head: DINOv2ProjectionHead, ibot_head: DINOv2ProjectionHead) -> None:
        super().__init__()
        self.dino_head = dino_head
        self.ibot_head = ibot_head


class _Wrapped(nn.Module):
    """EmbeddingModel.wrapped_model / DINOv2ViTModelWrapper._model naming shell (SURVEY.md appendix A)."""

    def __init__(self, model: DinoVisionTransformer) -> None:
        super().__init__()
        self._model = model

    def get_model(self) -> DinoVisionTransformer:
        return self._model

    def set_activation_checkpointing(self, enabled: bool, every_n_blocks: int = 1) -> None:
        """DINOv2ViTModelWrapper.set_activation_checkpointing (LT/_models/dinov2_vit/dinov2_vit.py:55-59)."""
        self._model._activation_checkpointing = enabled
        self._model._activation_checkpointing_every_n_blocks = every_n_blocks

    @torch.no_grad()
    def forward_features(self, x: Tensor, masks: Optional[Tensor] = None) -> Dict[str, Tensor]:
        """DINOv2ViTModelWrapper.forward_features (LT/_models/dinov2_vit/dinov2_vit.py:67-97)."""
        rt = self._model.forward_features(x, masks)
        pt = rt["x_norm_patchtokens"]
        b, _, d = pt.shape
        hh, ww = x.shape[2] // self._model.patch_size, x.shape[3] // self._model.patch_size
        return {"features": pt.permute(0, 2, 1).reshape(b, d, hh, ww), "cls_token": rt["x_norm_clstoken"]}


class _Embedding(nn.Module):
    def __init__(self, model: DinoVisionTransformer) -> None:
        super().__init__()
        self.wrapped_model = _Wrapped(model)


def _unwrap_backbone(embedding_model: Any) -> nn.Module:
    """EmbeddingModel(wrapped_model=DINOv2ViTModelWrapper(model)) | wrapper | the ViT itself -> the ViT."""
    m = embedding_model
    if hasattr(m, "wrapped_model"):
        m = m.wrapped_model
    if hasattr(m, "get_model"):
        m = m.get_model()
    return m


def backbone_kwargs_from_model(model: nn.Module) -> Dict[str, Any]:
    """Constructor arguments of a DinoVisionTransformer (the reference's or this package's) read back from the module."""
    blk0 = model.blocks[0]
    chunked = bool(getattr(model, "chunked_blocks", False))
    if chunked:  # BlockChunk(ModuleList): Identity padding then blocks (vision_transformer.py:215-226)
        blk0 = [b for b in blk0 if not isinstance(b, nn.Identity)][0]
    sd_names = [n for n, _ in model.named_parameters()]
    swiglu = any(".mlp.w12." in n for n in sd_names)
    ls = any(n.endswith("ls1.gamma") for n in sd_names)
    pe_w = model.patch_embed.proj.weight
    D = model.embed_dim
    hidden = dict(model.named_parameters())[[n for n in sd_names if n.endswith("mlp.w12.weight" if swiglu else "mlp.fc1.weight")][0]].shape[0]
    mlp_ratio = 4.0 if swiglu else hidden / D
    n_patches = model.pos_embed.shape[1] - 1
    # per-block stochastic-depth rates: reference Block keeps `sample_drop_ratio`, this package keeps `dpr`
    if hasattr(model, "dpr"):
        dpr = list(model.dpr)
    else:
        blocks = [b for c in model.blocks for b in (c if chunked else [c]) if not isinstance(b, nn.Identity)]
        dpr = [float(getattr(b, "sample_drop_ratio", 0.0)) for b in blocks]
    uniform = len(set(dpr)) == 1 and dpr[0] > 0
    gamma0 = None
    if ls:
        gamma0 = float(dict(model.named_parameters())[[n for n in sd_names if n.endswith("ls1.gamma")][0]].detach().flatten()[0]) or 1e-5
    return dict(img_size=int(round(n_patches ** 0.5)) * model.patch_size, patch_size=model.patch_size, in_chans=pe_w.shape[1],
                embed_dim=D, depth=model.n_blocks, num_heads=model.num_heads, mlp_ratio=mlp_ratio,
                drop_path_rate=max(dpr) if dpr else 0.0, drop_path_uniform=uniform, init_values=gamma0,
                ffn_layer="swiglu" if swiglu else "mlp", num_register_tokens=model.num_register_tokens,
                interpolate_antialias=model.interpolate_antialias, interpolate_offset=model.interpolate_offset)


def _unchunk(name: str) -> str:
    """`blocks.{chunk}.{i}.x` (block_chunks > 0 checkpoints) -> `blocks.{i}.x`."""
    parts = name.split(".")
    for j in range(len(parts) - 2):
        if parts[j] == "blocks" and parts[j + 1].isdigit() and parts[j + 2].isdigit():
            return ".".join(parts[:j + 1] + parts[j + 2:])
    return name


class DINOv2(nn.Module):
    def __init__(self, method_args: DINOv2Args, optimizer_args: DINOv2AdamWViTArgs, embedding_model: Any = None,
                 global_batch_size: int = 1024, num_input_channels: int = 3, *, model_kwargs: Optional[Dict[str, Any]] = None,
                 max_steps: int = 125_000, device: str = "cuda") -> None:
        """Same leading arguments as the reference (LT/_methods/dinov2/dinov2.py:179-186).  `embedding_model` is either
          * a pre-built backbone -- the reference's EmbeddingModel / DINOv2ViTModelWrapper / DinoVisionTransformer or this
            package's DinoVisionTransformer: its architecture is read back and its weights initialise teacher and student
            (the reference deep-copies the teacher into the student, :197-198), or
          * a dict of DinoVisionTransformer constructor arguments (embed_dim, depth, num_heads, patch_size, init_values,
            drop_path_rate, num_register_tokens, ...; what `dinov2/vits14-noreg` etc. resolve to); `model_kwargs=` is
            the keyword spelling of the same."""
        super().__init__()
        init_state = None
        if model_kwargs is None:
            if isinstance(embedding_model, dict):
                model_kwargs = embedding_model
            elif embedding_model is not None:
                bb = _unwrap_backbone(embedding_model)
                model_kwargs = backbone_kwargs_from_model(bb)
                init_state = {_unchunk(k): v.detach() for k, v in bb.state_dict().items()}
            else:
                raise ValueError("DINOv2 needs an embedding_model (module) or model_kwargs (dict)")
        if method_args.batch_norm:
            raise NotImplementedError("batch_norm heads are not implemented on the B200 path")
        self.method_args = method_args
        self.optimizer_args = optimizer_args
        self.global_batch_size = global_batch_size
        self.trainer = _TrainerState(max_steps)
        self.device_ = torch.device(device)
        a = method_args
        mk = dict(model_kwargs)
        mk.setdefault("in_chans", num_input_channels)
        probe = dict(img_size=mk.get("img_size", 224), patch_size=mk.get("patch_size", 16), embed_dim=mk["embed_dim"],
                     depth=mk["depth"], mlp_ratio=mk.get("mlp_ratio", 4.0))
        D = probe["embed_dim"]
        n_patches = (probe["img_size"] // probe["patch_size"]) ** 2
        shapes: Dict[str, Tuple[int, ...]] = {}
        swiglu = mk.get("ffn_layer", "mlp") != "mlp"
        hidden = int(D * probe["mlp_ratio"])
        if swiglu:
            hidden = (int(hidden * 2 / 3) + 7) // 8 * 8  # SwiGLUFFNFused hidden size (layers/swiglu_ffn.py:60-63)
        for k, v in vit_param_shapes(D, probe["depth"], probe["patch_size"], mk["in_chans"], n_patches,
                                     hidden, mk.get("num_register_tokens", 0),
                                     bool(mk.get("init_values")), swiglu).items():
            shapes["backbone." + k] = v
        hs = head_param_shapes(D, a.hidden_dim, a.dino_bottleneck_dim, a.output_dim)
        for k, v in hs.items():
            shapes["dino_head." + k] = v
        if a.ibot_separate_head:
            for k, v in hs.items():
                shapes["ibot_head." + k] = v
        self.s_arena = Arena(shapes, device, with_grad=True, with_optim_state=True)
        self.t_arena = Arena(shapes, device, with_grad=False, with_optim_state=False)

        def build(arena: Arena, train: bool):
            mkk = dict(mk)
            if not train:
                mkk["drop_path_rate"] = 0.0  # make_teacher(): teacher has no stochastic depth (dinov2_vit.py:108-151)
            vit = DinoVisionTransformer(**mkk, arena=arena, prefix="backbone.", requires_grad=train)
            dino = DINOv2ProjectionHead(D, a.output_dim, hidden_dim=a.hidden_dim, bottleneck_dim=a.dino_bottleneck_dim,
                                        arena=arena, prefix="dino_head.", requires_grad=train)
            ibot = dino
            if a.ibot_separate_head:
                ibot = DINOv2ProjectionHead(D, a.output_dim, hidden_dim=a.hidden_dim, bottleneck_dim=a.dino_bottleneck_dim,
                                            arena=arena, prefix="ibot_head.", requires_grad=train)
            return vit, dino, ibot

        s_vit, s_dino, s_ibot = build(self.s_arena, True)
        t_vit, t_dino, t_ibot = build(self.t_arena, False)
        # student = deepcopy(teacher) in the reference (dinov2.py:197-198); heads are initialised independently
        off, n = self.s_arena.offsets["dino_head.mlp.0.weight"]
        if init_state is not None:
            for k, v in init_state.items():
                if "backbone." + k in self.t_arena.offsets:
                    self.t_arena.p("backbone." + k).copy_(v.to(device, torch.float32).view(self.t_arena.shapes["backbone." + k]))
            self.t_arena.bf16_valid = False
        self.s_arena.fp32[:off].copy_(self.t_arena.fp32[:off])
        self.s_arena.bf16_valid = False
        self.teacher_embedding_model = _Embedding(t_vit)
        self.student_embedding_model = _Embedding(s_vit)
        self.teacher_head = DINOv2Head(t_dino, t_ibot)
        self.student_head = DINOv2Head(s_dino, s_ibot)
        self._patch_size = s_vit.patch_size
        self.dino_loss = DINOLoss(a.output_dim, a.student_temp, a.center_momentum).to(device)
        self.ibot_loss = IBOTPatchLoss(a.output_dim, a.student_temp, a.center_momentum).to(device)
        self._opt_step = 0
        self._optimizer: Optional["FusedAdamWEMA"] = None
        self._scheduler: Optional["CosineWarmupFactor"] = None
        self._ema_done = False
        # iBOT masks: "host" = the reference's python-`random` generator (bit-exact stream, default); "device" = csrc/masks.cu
        self.mask_source = "host"
        self.mask_seed = 0
        self._mask_step_dev: Optional[Tensor] = None
        self.debug_taps: Optional[Dict[str, Any]] = None
        self.logged: Dict[str, Any] = {}
        self._last_result: Optional[TrainingStepResult] = None
        self._build_optimizer_tables()
        # weights written through load_state_dict() land in the fp32 arenas: the bf16 GEMM shadows of BOTH sides are stale
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._invalidate_shadows())
        # KoLeo runs one CTA per crop group with the group's features in shared memory (csrc/loss.cu)
        D_ = s_vit.embed_dim
        self._koleo_max_batch = (220 * 1024 // 4) // (2 * D_ + 3)
        self._grad_ready = False
        self._seg_cache: Dict[Tuple[int, int, int], Tensor] = {}
        self._static: Optional[Dict[str, Any]] = None
        self.use_cuda_graph = False

    def _invalidate_shadows(self) -> None:
        self.s_arena.bf16_valid = False
        self.t_arena.bf16_valid = False

    # ------------------------------------------------------------------ accessors
    @property
    def s_vit(self) -> DinoVisionTransformer:
        return self.student_embedding_model.wrapped_model._model

    @property
    def t_vit(self) -> DinoVisionTransformer:
        return self.teacher_embedding_model.wrapped_model._model

    # ------------------------------------------------------------------ optimizer tables (configure_optimizers :550-586)
    def _build_optimizer_tables(self) -> None:
        a = self.method_args
        lr_scale = a.reference_batch_size and self.global_batch_size / a.reference_batch_size
        if a.lr_scale_method == "sqrt":
            lr_scale = math.sqrt(lr_scale)
        self.base_lr = self.optimizer_args.lr * lr_scale
        nl = self.s_vit.n_blocks
        lr_t, wd_t, fl_t = {}, {}, {}
        for name in self.s_arena.names():
            if name.startswith("backbone."):
                st = param_group_settings(name[len("backbone."):], True, nl, a.layerwise_decay, a.patch_embed_lr_multiplier)
                flags = 2  # bit1: "head" not in group name -> frozen by student_freeze_backbone_steps
            else:
                # parameters of DINOv2Head are named "dino_head.*" / "ibot_head.*" inside trainable_modules()
                st = param_group_settings(name, False, nl, a.layerwise_decay, a.patch_embed_lr_multiplier)
                flags = 1 if st["last_layer"] else 0
            lr_t[name], wd_t[name], fl_t[name] = st["lr_scale"], st["wd_scale"], flags
        self.lr_table = self.s_arena.chunk_table(lr_t)
        self.wd_table = self.s_arena.chunk_table(wd_t)
        self.flag_table = self.s_arena.chunk_table(fl_t, dtype=torch.uint8)
        self.weight_decay_start = (self.optimizer_args.weight_decay if a.weight_decay_start == "auto"
                                   else float(a.weight_decay_start))
        self.gradnorm_sq = torch.zeros(1, device=self.device_, dtype=torch.float32)
        self._side_stream = torch.cuda.Stream(device=self.device_) if self.device_.type == "cuda" else None
        self._comm_stream = torch.cuda.Stream(device=self.device_) if self.device_.type == "cuda" else None
        self._head_ready = torch.cuda.Event() if self.device_.type == "cuda" else None
        self._mid_ready = torch.cuda.Event() if self.device_.type == "cuda" else None
        self._head_work = None
        self._mid_work = None
        self.force_backbone_split: Optional[int] = None  # tests: cut the backbone backward at this block on a single rank
        self._head_off = self.s_arena.offsets["dino_head.mlp.0.weight"][0]  # arena order: backbone.*, then the heads

    # ------------------------------------------------------------------ the step
    def _allreduce_head_grads_async(self) -> None:
        """Data-parallel runs: start the all-reduce of the projection-head gradients (the arena's tail, ~half of all
        parameters; final once the head backward has run) on a communication stream, so that it overlaps the backbone
        backward.  `optimizer_step` reduces the backbone part and waits for this one."""
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            return
        main = torch.cuda.current_stream()
        self._head_ready.record(main)
        self._comm_stream.wait_event(self._head_ready)
        with torch.cuda.stream(self._comm_stream):
            self._head_work = dist.all_reduce(self.s_arena.grad[self._head_off:], async_op=True)

    def _backbone_split(self) -> int:
        """Block index at which the backbone backward is cut for the second overlapped all-reduce (0: no cut)."""
        nb = self.s_vit.n_blocks
        if self.force_backbone_split is not None:
            return self.force_backbone_split
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        # a single rank has nothing to overlap: no cut, one graph fewer
        return max(1, int(nb * DDP_SPLIT_FRAC)) if (nb >= 4 and multi) else 0

    def _allreduce_upper_backbone_async(self, split_at: int) -> None:
        """Data-parallel runs: all-reduce the gradients of blocks >= split_at and of `norm` (contiguous in the arena, final
        after `_core_b(split_at=...)`) on the communication stream while `_core_b2` runs."""
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            return
        lo = self.s_arena.offsets[f"backbone.blocks.{split_at}.norm1.weight"][0]
        hi = self.s_arena.offsets["backbone.mask_token"][0]  # arena order: ..., blocks.*, norm.*, mask_token, heads
        main = torch.cuda.current_stream()
        self._mid_ready.record(main)
        self._comm_stream.wait_event(self._mid_ready)
        with torch.cuda.stream(self._comm_stream):
            self._mid_work = (dist.all_reduce(self.s_arena.grad[lo:hi], async_op=True), lo, hi)

    def _masks(self, n_crops: int, h: int, w: int):
        a = self.method_args
        gen = MaskingGenerator(input_size=(h, w), max_num_patches=int(0.5 * h * w))
        return create_collated_masks(a.mask_ratio_min, a.mask_ratio_max, int(n_crops * a.mask_probability), n_crops, gen)

    def _mask_targets(self, n_crops: int, n_tokens: int) -> List[int]:
        """Per-crop mask counts exactly as create_collated_masks draws them (utils.py:116-133): one uniform draw per masked
        crop inside its ratio bucket, zero for the others, then the shuffle -- a few dozen python-`random` draws per step."""
        import random

        import numpy as np

        a = self.method_args
        n_masked = int(n_crops * a.mask_probability)
        edges = np.linspace(a.mask_ratio_min, a.mask_ratio_max, n_masked + 1)
        t = [int(n_tokens * random.uniform(edges[i], edges[i + 1])) for i in range(n_masked)] + [0] * (n_crops - n_masked)
        random.shuffle(t)
        return t

    def _device_masks(self, n_crops: int, h: int, w: int, bufs: Optional[Dict[str, Tensor]] = None) -> Dict[str, Any]:
        """Block-wise masks generated ON THE DEVICE (csrc/masks.cu): only the per-crop target counts come from the host.
        Returns padded, static-shape tensors (capacity = the targets' sum rounded up to 512): rows >= M are inert."""
        dev = self.device_
        targets = self._mask_targets(n_crops, h * w)
        cap = max(512, -(-sum(targets) // 512) * 512)
        if bufs is None:
            bufs = {"targets": torch.empty(n_crops, device=dev, dtype=torch.int32),
                    "masks_u8": torch.empty(n_crops, h * w, device=dev, dtype=torch.uint8),
                    "idx": torch.empty(cap, device=dev, dtype=torch.int64), "mw": torch.empty(cap, device=dev),
                    "iw": torch.empty(cap, device=dev), "pad": torch.empty(cap, device=dev),
                    "m_valid": torch.empty(1, device=dev, dtype=torch.int32)}
        if self._mask_step_dev is None:
            self._mask_step_dev = torch.zeros(1, device=dev, dtype=torch.int32)
        bufs["targets"].copy_(torch.tensor(targets, dtype=torch.int32), non_blocking=True)
        ops.block_masks(bufs["targets"], h, w, int(0.5 * h * w), self.mask_seed, bufs["masks_u8"], step_dev=self._mask_step_dev)
        ops.collate_masks(bufs["masks_u8"], cap, bufs["idx"], bufs["mw"], bufs["iw"], bufs["pad"], bufs["m_valid"])
        self._mask_step_dev.add_(1)
        return {"device": True, "cap": cap, "collated_masks_u8": bufs["masks_u8"], "mask_indices_list": bufs["idx"][:cap],
                "masks_weight": bufs["mw"][:cap], "row_w": bufs["iw"][:cap], "pad": bufs["pad"][:cap], "m_valid": bufs["m_valid"]}

    def training_step_impl(self, batch: Dict[str, Any], batch_idx: int = 0) -> TrainingStepResult:
        """Loss evaluation + explicit backward (gradients land in the arena / `param.grad`). Eager launch schedule."""
        # the kernels take raw device pointers: a model built in host memory fails here, before any launch (with a GPU
        # present such a launch would fault asynchronously and leave the CUDA context unusable)
        ops._req_cuda(self.s_arena.fp32)
        a = self.method_args
        dev = self.device_
        teacher_temp = linear_warmup_schedule(self.trainer.global_step, a.teacher_temp_warmup_steps,
                                              a.teacher_temp_start, a.teacher_temp_end)
        views: List[Tensor] = batch["views"]
        gv = torch.cat(views[:2])
        lv = torch.cat(views[2:]) if len(views) > 2 else None
        p = self._patch_size
        masks = batch.get("masks")
        if masks is None:
            if self.mask_source == "device":
                masks = self._device_masks(gv.shape[0], gv.shape[2] // p, gv.shape[3] // p)
            else:
                masks = self._masks(gv.shape[0], gv.shape[2] // p, gv.shape[3] // p)  # host python RNG, reference stream
        for arena in (self.s_arena, self.t_arena):
            if not arena.bf16_valid:
                arena.refresh_bf16()
        if a.center_method == "softmax":
            self.dino_loss.apply_center_update()
            self.ibot_loss.apply_center_update()
        if masks.get("device"):  # padded static-shape mask tensors produced on the device: rows >= M are inert
            mask_idx = masks["mask_indices_list"]
            st = self._core_a(gv, lv, masks["collated_masks_u8"], mask_idx, masks["masks_weight"], 1.0 / teacher_temp, None,
                              masks["row_w"], masks["m_valid"], masks["pad"])
        else:
            collated = masks["collated_masks"].to(dev, non_blocking=True)
            mask_idx = masks["mask_indices_list"].to(dev, non_blocking=True)
            masks_weight = masks["masks_weight"].to(dev, torch.float32, non_blocking=True)
            st = self._core_a(gv, lv, collated.to(torch.uint8), mask_idx, masks_weight, 1.0 / teacher_temp, None, None, None)
        self._allreduce_head_grads_async()
        split_at = self._backbone_split()
        out = self._core_b(st, split_at)
        if split_at > 0:
            self._allreduce_upper_backbone_async(split_at)
            out = self._core_b2(st)
        if a.center_method == "softmax":
            self.dino_loss._launch_reduce(out["dino_center_sum"], gv.shape[0])
            if mask_idx.shape[0]:
                self.ibot_loss._launch_reduce(out["ibot_center_sum"], 1)
        return self._result(out)

    def _result(self, out: Dict[str, Tensor]) -> TrainingStepResult:
        a = self.method_args
        lt, koleo = out["loss_terms"], out["koleo"]
        dino_global, dino_local, ibot = lt[0], lt[1], lt[2]
        koleo_loss = koleo.sum()
        loss = (a.dino_loss_weight * dino_global + a.dino_loss_weight * dino_local + a.ibot_loss_weight * ibot
                + a.koleo_loss_weight * koleo_loss)
        self._grad_ready = True
        return TrainingStepResult(loss=loss, log_dict={
            "train_loss/dino_global_loss": dino_global, "train_loss/dino_local_loss": dino_local,
            "train_loss/ibot_loss": ibot, "train_loss/koleo_loss": koleo_loss})

    def _core_a(self, gv: Tensor, lv: Optional[Tensor], masks_u8: Tensor, mask_idx: Tensor, masks_weight: Tensor,
                t_scale: float, t_scale_dev: Optional[Tensor], ibot_rowvec: Optional[Tensor],
                m_valid_dev: Optional[Tensor], pad_mask: Optional[Tensor] = None) -> Dict[str, Any]:
        """First half of the device schedule of one step: teacher, student forward, losses, HEAD backward.  When it
        returns, the gradients of the projection heads (the tail of the flat arena, half of all parameters) are final,
        so their all-reduce can overlap `_core_b` (the backbone backward).  Shapes depend only on the arguments' shapes, every per-step scalar is
        either a kernel argument (eager) or read from device memory (`*_dev`), and no host<->device traffic or
        synchronisation happens inside -- so the whole function can be captured into a CUDA graph.
        With padding (graph mode) rows >= *m_valid_dev of mask_idx/masks_weight are inert (weight 0)."""
        a = self.method_args
        dev = self.device_
        n_global = 2
        n_crops = gv.shape[0]
        B = n_crops // n_global
        LB = lv.shape[0] if lv is not None else 0
        n_local = LB // B
        g_terms = (n_global - 1) * n_global
        l_terms = max(n_local * n_global, 1)
        p = self._patch_size
        hh, ww = gv.shape[2] // p, gv.shape[3] // p
        M = int(mask_idx.shape[0])
        s_vit, t_vit = self.s_vit, self.t_vit
        s_dino, s_ibot = self.student_head.dino_head, self.student_head.ibot_head
        t_dino, t_ibot = self.teacher_head.dino_head, self.teacher_head.ibot_head
        separate = a.ibot_separate_head
        D, K = s_vit.embed_dim, a.output_dim
        R = s_vit.num_register_tokens
        bf, f32 = torch.bfloat16, torch.float32
        for hd in {id(x): x for x in (s_dino, s_ibot, t_dino, t_ibot)}.values():
            hd.refresh_last_layer()
        self.s_arena.zero_grad()
        out: Dict[str, Tensor] = {}

        # ---------------- teacher (dinov2.py:399-472)
        tctx = t_vit._fwd(gv, None, save=False)
        Ng = tctx.dims[3]
        cls_rows = torch.arange(n_crops, device=dev, dtype=torch.int64) * Ng
        cls_rows_swapped = torch.cat([cls_rows[B:], cls_rows[:B]])  # A<->B swap (:415-417)
        t_in = torch.empty(n_crops + M, D, device=dev, dtype=bf)
        ops.gather_rows(tctx.xnorm, cls_rows_swapped, t_in[:n_crops])
        ops.gather_rows(tctx.xnorm, mask_idx, t_in[n_crops:], Np=hh * ww, N=Ng, off=1 + R)
        t_logits = torch.empty(n_crops + M, K, device=dev, dtype=bf)
        if separate:
            t_dino._fwd(t_in[:n_crops], save=False, logits=t_logits[:n_crops])
            if M:
                t_ibot._fwd(t_in[n_crops:], save=False, logits=t_logits[n_crops:])
        else:
            t_dino._fwd(t_in, save=False, logits=t_logits)
        del tctx
        t_rowterm = torch.empty(n_crops + M, device=dev, dtype=f32)
        colterm_d = torch.empty(K, device=dev, dtype=f32)
        colterm_i = torch.empty(K, device=dev, dtype=f32)
        if a.center_method == "softmax":
            ops.vec_op(colterm_d, self.dino_loss.center.view(-1), t_scale, 0.0, 1, a_dev=t_scale_dev)
            ops.vec_op(colterm_i, self.ibot_loss.center.view(-1), t_scale, 0.0, 1, a_dev=t_scale_dev)
            # per-rank center batch sums (reduce_center_update, dinov2_loss.py:139-145 / :274-282)
            out["dino_center_sum"] = torch.zeros(K, device=dev, dtype=f32)
            ops.col_reduce(t_logits[:n_crops], out["dino_center_sum"])
            out["ibot_center_sum"] = torch.zeros(K, device=dev, dtype=f32)
            if M:
                rv = ibot_rowvec if ibot_rowvec is not None else torch.full((M,), 1.0 / M, device=dev, dtype=f32)
                ops.col_reduce(t_logits[n_crops:], out["ibot_center_sum"], rowvec=rv)
        elif a.center_method == "sinkhorn_knopp":
            # (with several ranks the prototype sums are all-reduced inside sinkhorn_colterm; under graph capture those NCCL
            # kernels become part of the step graph, see `_graph_ok`)
            colterm_d = sinkhorn_colterm(t_logits[:n_crops], t_scale, scale_dev=t_scale_dev)
            if M:
                colterm_i = sinkhorn_colterm(t_logits[n_crops:], t_scale, scale_dev=t_scale_dev, row_mask=pad_mask)
        else:
            raise ValueError(f"Unknown centering method: {a.center_method}")
        ops.row_lse(t_logits[:n_crops], colterm_d, t_scale, t_rowterm[:n_crops], scale_dev=t_scale_dev)
        # (the masked-patch rows' teacher log-sum-exp is computed inside the CE kernel: one HBM read of those logits)

        # ---------------- student forward (dinov2.py:474-519)
        sg = s_vit._fwd(gv, masks_u8, save=True, drop_path=True)
        sl = None
        lcls_rows = None
        if lv is not None:
            sl = s_vit._fwd(lv, None, save=True, drop_path=True)
        Rs = n_crops + LB + M
        s_in = torch.empty(Rs, D, device=dev, dtype=bf)
        ops.gather_rows(sg.xnorm, cls_rows, s_in[:n_crops])
        if sl is not None:
            Nl = sl.dims[3]
            lcls_rows = torch.arange(LB, device=dev, dtype=torch.int64) * Nl
            ops.gather_rows(sl.xnorm, lcls_rows, s_in[n_crops:n_crops + LB])
        ops.gather_rows(sg.xnorm, mask_idx, s_in[n_crops + LB:], Np=hh * ww, N=Ng, off=1 + R)
        s_logits = torch.empty(Rs, K, device=dev, dtype=bf)
        nd = n_crops + LB
        if separate:
            hc_d = s_dino._fwd(s_in[:nd], save=True, logits=s_logits[:nd])
            hc_i = s_ibot._fwd(s_in[nd:], save=True, logits=s_logits[nd:]) if M else None
        else:
            hc_d = s_dino._fwd(s_in, save=True, logits=s_logits)
            hc_i = None

        # ---------------- fused CE forward + backward
        terms = g_terms + l_terms
        idx0 = torch.empty(Rs, device=dev, dtype=torch.int32)
        idx1 = torch.full((Rs,), -1, device=dev, dtype=torch.int32)
        wrow = torch.empty(Rs, device=dev, dtype=f32)
        idx0[:n_crops] = torch.arange(n_crops, device=dev, dtype=torch.int32)
        wrow[:n_crops] = (1.0 / n_crops) * 2.0 / terms
        if LB:
            bidx = torch.arange(LB, device=dev, dtype=torch.int32) % B
            idx0[n_crops:nd] = bidx
            idx1[n_crops:nd] = bidx + B
            wrow[n_crops:nd] = (1.0 / B) / terms
        if M:
            idx0[nd:] = torch.arange(M, device=dev, dtype=torch.int32)
            wrow[nd:] = masks_weight / n_crops
        loss_rows = torch.empty(Rs, device=dev, dtype=f32)
        ds = torch.empty(Rs, K, device=dev, dtype=bf)
        s_scale = 1.0 / a.student_temp
        ops.dino_ce(s_logits[:nd], t_logits[:n_crops], colterm_d, t_rowterm[:n_crops], idx0[:nd], idx1[:nd], wrow[:nd],
                    s_scale, t_scale, loss_rows[:nd], ds[:nd], gscale=a.dino_loss_weight, t_scale_dev=t_scale_dev)
        if M:
            ops.dino_ce(s_logits[nd:], t_logits[n_crops:], colterm_i, None, idx0[nd:], None, wrow[nd:],
                        s_scale, t_scale, loss_rows[nd:], ds[nd:], gscale=a.ibot_loss_weight, t_scale_dev=t_scale_dev)
        seg = self._segments(n_crops, nd, Rs)
        loss_terms = torch.zeros(3, device=dev, dtype=f32)
        ops.segment_sum(loss_rows, seg, loss_terms)
        if self.debug_taps is not None:  # tests / bench parity read the head outputs (bf16 logits) of this step
            self.debug_taps.update(t_logits=t_logits.clone(), s_logits=s_logits.clone(), n_crops=n_crops, n_local_rows=LB, n_masked=M)
        del s_logits, t_logits

        # ---------------- head backward -> gradient wrt the backbone outputs
        dxn_g = torch.zeros(sg.dims[4], D, device=dev, dtype=f32)
        if separate:
            dx_d = s_dino._bwd(hc_d, ds[:nd])
            dx_i = s_ibot._bwd(hc_i, ds[nd:]) if M else None
        else:
            dx_all = s_dino._bwd(hc_d, ds)
            dx_d, dx_i = dx_all[:nd], dx_all[nd:]
        ops.scatter_rows(dx_d[:n_crops], cls_rows, dxn_g)
        if M:
            ops.scatter_rows(dx_i, mask_idx, dxn_g, Np=hh * ww, N=Ng, off=1 + R, count_dev=m_valid_dev)
        return dict(out=out, loss_terms=loss_terms, sg=sg, sl=sl, dx_d=dx_d, dxn_g=dxn_g, n_crops=n_crops, B=B, Ng=Ng,
                    lcls_rows=lcls_rows)

    def _core_b(self, st: Dict[str, Any], split_at: int = 0) -> Dict[str, Tensor]:
        """Second half: KoLeo and the backbone backward (local crops, then global crops).  split_at > 0 stops the
        global-crop backward before block `split_at - 1` (continued by `_core_b2`)."""
        a = self.method_args
        dev = self.device_
        f32 = torch.float32
        s_vit = self.s_vit
        D = s_vit.embed_dim
        # pop: the activation contexts must die with the local names below (the local-crop activations are released
        # before the global-crop backward runs)
        out, loss_terms, sg, sl, dx_d, dxn_g = (st.pop(k) for k in ("out", "loss_terms", "sg", "sl", "dx_d", "dxn_g"))
        n_crops, B, Ng, lcls_rows = st["n_crops"], st["B"], st["Ng"], st["lcls_rows"]
        # KoLeo on the pre-head global cls tokens (:377-380): forward value + gradient (+=) into dxn_g
        koleo = torch.zeros(2, device=dev, dtype=f32)
        if B < 2:
            raise _lib.B200Error("KoLeo needs at least 2 images per GPU (nearest neighbour inside the crop group)")
        # two CTAs of pure latency (~160 us): forked onto a side stream (a parallel branch of the captured graph) so it
        # overlaps the local-crop backward; its += into dxn_g is only needed by the global-crop backward below
        main = torch.cuda.current_stream()
        side = self._side_stream if sl is not None else None
        if side is not None:
            side.wait_stream(main)
        with torch.cuda.stream(side if side is not None else main):
            ops.koleo(sg.xnorm.view(n_crops, Ng, D)[:, 0], 2, B, koleo, dxn_g.view(n_crops, Ng, D)[:, 0],
                      gscale=a.koleo_loss_weight)
        if sl is not None:
            dxn_l = torch.zeros(sl.dims[4], D, device=dev, dtype=f32)
            ops.scatter_rows(dx_d[n_crops:], lcls_rows, dxn_l)
            s_vit._bwd(sl, dxn_l)
            del sl, dxn_l
        if side is not None:
            main.wait_stream(side)
        out["loss_terms"], out["koleo"] = loss_terms, koleo
        if split_at <= 0:
            s_vit._bwd(sg, dxn_g)
            return out
        # first segment of the global-crop backward: final LayerNorm + blocks nb-1 .. split_at.  When it returns, the
        # gradients of those blocks and of `norm` are final (the local-crop pass above already added its share): their
        # all-reduce overlaps `_core_b2`
        st["bwd_state"] = s_vit._bwd(sg, dxn_g, stop_before=split_at)
        st["sg"], st["out"] = sg, out
        return out

    def _core_b2(self, st: Dict[str, Any]) -> Dict[str, Tensor]:
        """Last segment: global-crop backward of blocks split-1 .. 0 and the embeddings."""
        sg, state = st.pop("sg"), st.pop("bwd_state")
        self.s_vit._bwd(sg, None, state=state)
        return st.pop("out")

    def _segments(self, n_crops: int, nd: int, Rs: int) -> Tensor:
        key = (n_crops, nd, Rs)
        if key not in self._seg_cache:
            self._seg_cache[key] = torch.tensor([0, n_crops, nd, Rs], device=self.device_, dtype=torch.int32)
        return self._seg_cache[key]

    # ------------------------------------------------------------------ CUDA-graph replay of the step
    def _graphed_step(self, batch: Dict[str, Any]) -> TrainingStepResult:
        """Same arithmetic as training_step_impl, replayed from a captured CUDA graph (one graph per padded
        masked-token count, bucketed to 512): ~1000 kernel launches per step leave the host's critical path."""
        a = self.method_args
        dev = self.device_
        views: List[Tensor] = batch["views"]
        B = views[0].shape[0]
        n_local = len(views) - 2
        p = self._patch_size
        hh, ww = views[0].shape[2] // p, views[0].shape[3] // p
        st = self._static
        if st is None or st["key"] != (B, n_local, tuple(views[0].shape[1:]), tuple(views[-1].shape[1:])):
            cap_max = max(512, -(-(int(2 * B * a.mask_probability) * int(0.5 * hh * ww)) // 512) * 512)
            st = self._static = {
                "key": (B, n_local, tuple(views[0].shape[1:]), tuple(views[-1].shape[1:])),
                "gv": torch.empty(2 * B, *views[0].shape[1:], device=dev),
                "lv": torch.empty(n_local * B, *views[-1].shape[1:], device=dev) if n_local else None,
                "masks_u8": torch.zeros(2 * B, hh * ww, device=dev, dtype=torch.uint8),
                "idx": torch.zeros(cap_max, device=dev, dtype=torch.int64),
                "mw": torch.zeros(cap_max, device=dev, dtype=torch.float32),
                "iw": torch.zeros(cap_max, device=dev, dtype=torch.float32),
                "pad": torch.zeros(cap_max, device=dev, dtype=torch.float32),
                "m_valid": torch.zeros(1, device=dev, dtype=torch.int32),
                "t_scale": torch.zeros(1, device=dev, dtype=torch.float32),
                "graphs": {}, "pool": None, "cap_max": cap_max,
            }
        teacher_temp = linear_warmup_schedule(self.trainer.global_step, a.teacher_temp_warmup_steps,
                                              a.teacher_temp_start, a.teacher_temp_end)
        masks = batch.get("masks")
        # stage the step's inputs into the static buffers (device copies for resident views, H2D otherwise)
        for i in range(2):
            st["gv"][i * B:(i + 1) * B].copy_(views[i], non_blocking=True)
        for i in range(n_local):
            st["lv"][i * B:(i + 1) * B].copy_(views[2 + i], non_blocking=True)
        if masks is None and self.mask_source == "device":
            # masks, index list, weights and padding masks are written straight into the static buffers by two kernels
            if "targets" not in st:
                st["targets"] = torch.empty(2 * B, device=dev, dtype=torch.int32)
            cap = self._device_masks(2 * B, hh, ww, bufs=st)["cap"]
        else:
            if masks is None:
                masks = self._masks(2 * B, hh, ww)
            M = int(masks["mask_indices_list"].shape[0])
            cap = max(512, -(-M // 512) * 512)
            if a.center_method != "softmax" and _world_size() > 1:
                # the captured Sinkhorn all-reduces must be replayed by every rank every step: one shape for all ranks and
                # steps (the masked-token count differs per rank), i.e. the guaranteed upper bound
                cap = max(cap, st["cap_max"])
            st["masks_u8"].copy_(masks["collated_masks"].to(torch.uint8), non_blocking=True)
            idx_h = torch.zeros(cap, dtype=torch.int64); idx_h[:M] = masks["mask_indices_list"]
            mw_h = torch.zeros(cap, dtype=torch.float32); mw_h[:M] = masks["masks_weight"]
            iw_h = torch.zeros(cap, dtype=torch.float32); iw_h[:M] = 1.0 / max(M, 1)
            st["idx"][:cap].copy_(idx_h, non_blocking=True)
            st["mw"][:cap].copy_(mw_h, non_blocking=True)
            st["iw"][:cap].copy_(iw_h, non_blocking=True)
            pad_h = torch.full((cap,), -1e30, dtype=torch.float32); pad_h[:M] = 0.0
            st["pad"][:cap].copy_(pad_h, non_blocking=True)
            st["m_valid"].fill_(M)
        st["t_scale"].fill_(1.0 / teacher_temp)
        for arena in (self.s_arena, self.t_arena):
            if not arena.bf16_valid:
                arena.refresh_bf16()
        if a.center_method == "softmax":
            self.dino_loss.apply_center_update()
            self.ibot_loss.apply_center_update()

        def run_a() -> Dict[str, Any]:
            return self._core_a(st["gv"], st["lv"], st["masks_u8"], st["idx"][:cap], st["mw"][:cap], 0.0, st["t_scale"],
                                st["iw"][:cap], st["m_valid"], st["pad"][:cap])

        split_at = self._backbone_split()
        entry = st["graphs"].get(cap)
        if entry is None:
            warm = run_a()  # eager warm-up at this shape (no collective: ranks reach new shapes at different steps)
            self._core_b(warm, split_at)
            if split_at > 0:
                self._core_b2(warm)
            del warm
            torch.cuda.synchronize()
            # three graphs sharing one memory pool: [teacher, student fwd, losses, head bwd] | [local-crop backward, upper
            # half of the global-crop backward] | [lower half + embeddings]; the all-reduce of the gradients that are final
            # after each graph is issued between the replays and overlaps the next one
            g1, g2, g3 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            if a.center_method != "softmax" and _world_size() > 1:  # graph 1 will hold captured all-reduces
                _NCCL_GRAPH_HOLDERS.add(self)
                _hook_process_group_teardown()
            n0 = _lib.LAUNCHES
            with torch.cuda.graph(g1, pool=st["pool"], capture_error_mode="thread_local"):  # NCCL watchdog thread may touch CUDA
                mid = run_a()
            if st["pool"] is None:
                st["pool"] = g1.pool()
            with torch.cuda.graph(g2, pool=st["pool"], capture_error_mode="thread_local"):
                outs = self._core_b(mid, split_at)
            if split_at > 0:
                with torch.cuda.graph(g3, pool=st["pool"], capture_error_mode="thread_local"):
                    outs = self._core_b2(mid)
            else:
                g3 = None
            n_captured = _lib.LAUNCHES - n0
            _lib.LAUNCHES = n0  # captured, not executed; every replay executes all of them
            entry = st["graphs"][cap] = (g1, g2, g3, outs, n_captured)
        g1, g2, g3, outs, n_captured = entry
        g1.replay()
        self._allreduce_head_grads_async()
        g2.replay()
        if g3 is not None:
            self._allreduce_upper_backbone_async(split_at)
            g3.replay()
        _lib.LAUNCHES += n_captured
        if a.center_method == "softmax":
            self.dino_loss._launch_reduce(outs["dino_center_sum"], 2 * B)
            self.ibot_loss._launch_reduce(outs["ibot_center_sum"], 1)
        return self._result(outs)

    # ------------------------------------------------------------------ Method surface (LT/_methods/method.py:131-148)
    def training_step(self, batch: Dict[str, Any], batch_idx: int = 0) -> Tensor:
        """Method.training_step: run the step, log `train_loss` + the log_dict with sync_dist=True semantics (cross-rank
        mean; ONE tiny all-reduce for all five scalars), return the loss."""
        if self._graph_ok():
            res = self._graphed_step(batch)
        else:
            res = self.training_step_impl(batch, batch_idx)
        self._last_result = res
        names = ["train_loss"] + list(res.log_dict.keys())
        vals = torch.stack([res.loss.reshape(())] + [v.reshape(()) for v in res.log_dict.values()])
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            vals = vals / dist.get_world_size()
            dist.all_reduce(vals)
        for k, v in zip(names, vals.unbind(0)):
            self.log(k, v, sync_dist=False)
        return res.loss

    def log(self, name: str, value: Any, **kwargs: Any) -> None:
        """Stand-in for LightningModule.log: keeps the latest value (a device scalar; no host sync) in `self.logged`."""
        self.logged[name] = value

    def log_dict(self, dictionary: Dict[str, Any], **kwargs: Any) -> None:
        for k, v in dictionary.items():
            self.log(k, v, **kwargs)

    def trainable_modules(self) -> List[nn.Module]:
        """LT/_methods/dinov2/dinov2.py:538-548."""
        return [self.student_embedding_model.wrapped_model.get_model(), self.student_head]

    # ------------------------------------------------------------------ optimizer + hooks (:550-660)
    def configure_optimizers(self):
        """([optimizer], [{"scheduler", "interval": "step"}]) like the reference (:550-586).  The optimizer is a shim over
        the fused sweep (clip + AdamW + EMA teacher + bf16 shadows in one kernel); its param_groups list one group per
        distinct (lr multiplier, weight-decay switch, freeze class), named after the group's first parameter as
        get_fused_param_groups does (utils.py:253-273)."""
        if self._optimizer is None:
            self._optimizer = FusedAdamWEMA(self)
            self._scheduler = CosineWarmupFactor(self)
        return [self._optimizer], [{"scheduler": self._scheduler, "interval": "step"}]

    def configure_gradient_clipping(self, optimizer: "FusedAdamWEMA", gradient_clip_val: Optional[float] = None,
                                    gradient_clip_algorithm: Optional[str] = None) -> None:
        """:588-598 -- clip_grad_norm_(method_args.gradient_clip_val); applied inside the sweep from the summed squares."""
        optimizer.clip_val = self.method_args.gradient_clip_val

    def on_before_optimizer_step(self, optimizer: "FusedAdamWEMA", *args: Any) -> None:
        """:600-639 -- cosine weight-decay schedule, backbone / last-layer lr freeze for the step about to run."""
        a = self.method_args
        step = self.trainer.global_step
        optimizer.weight_decay = cosine_schedule(step, self.trainer.estimated_stepping_batches, self.weight_decay_start,
                                                 a.weight_decay_end)
        optimizer.freeze_backbone = step < a.student_freeze_backbone_steps
        optimizer.freeze_last_layer = step < a.student_freeze_last_layer_steps
        optimizer.sync_param_groups()

    def on_train_batch_end(self, outputs: Any = None, batch: Any = None, batch_idx: int = 0) -> None:
        """:641-660 -- EMA teacher update with momentum cosine_schedule(trainer.global_step) (Lightning has already
        incremented global_step when this hook runs).  The fused sweep normally did it with that same momentum
        (`optimizer.step()`); this hook only does the work if the sweep ran without the EMA part."""
        if self._ema_done:
            self._ema_done = False
            return
        m = cosine_schedule(self.trainer.global_step, self.trainer.estimated_stepping_batches,
                            self.method_args.momentum_start, self.method_args.momentum_end)
        update_momentum(self.student_embedding_model, self.teacher_embedding_model, m)
        update_momentum(self.student_head, self.teacher_head, m)

    def optimizer_step(self) -> None:
        """What Lightning's automatic optimisation does after backward, in its hook order: on_before_optimizer_step ->
        configure_gradient_clipping -> optimizer.step -> scheduler.step -> global_step += 1 -> on_train_batch_end."""
        if not self._grad_ready:
            raise RuntimeError("optimizer_step() called without gradients; call training_step_impl first")
        (opt,), (sch,) = self.configure_optimizers()
        self.on_before_optimizer_step(opt)
        self.configure_gradient_clipping(opt)
        opt.step()
        sch["scheduler"].step()
        self.trainer.global_step += 1
        self.on_train_batch_end(None, None, 0)

    def _finish_grad_allreduce(self) -> None:
        """DDP gradient all-reduce (sum; the mean is folded into the sweep's grad_scale): reduce whatever part of the arena
        is not already in flight and make the current stream wait for the parts that are (the host never blocks)."""
        if self._head_work is not None:
            # the head part (and, when the backward was cut, blocks >= split and `norm`) are already in flight
            if self._mid_work is not None:
                work, lo, hi = self._mid_work
                dist.all_reduce(self.s_arena.grad[:lo])
                dist.all_reduce(self.s_arena.grad[hi:self._head_off])  # mask_token
                work.wait()
                self._mid_work = None
            else:
                dist.all_reduce(self.s_arena.grad[:self._head_off])
            self._head_work.wait()
            self._head_work = None
        else:
            dist.all_reduce(self.s_arena.grad)

    def _fused_sweep(self, opt: "FusedAdamWEMA", lr: float, fuse_ema: bool = True) -> None:
        """all-reduce(grad) -> deterministic sum of squares -> ONE sweep: clip + AdamW (per-chunk lr/wd, freezes) + EMA
        teacher + bf16 shadows of student and teacher."""
        a = self.method_args
        max_steps = self.trainer.estimated_stepping_batches
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        if world > 1:
            self._finish_grad_allreduce()
        ops.fill_f32(self.gradnorm_sq, 0.0)
        ops.sumsq(self.s_arena.grad, self.gradnorm_sq)
        # on_train_batch_end runs after Lightning has incremented global_step: the momentum index is step + 1
        momentum = cosine_schedule(self.trainer.global_step + 1, max_steps, a.momentum_start, a.momentum_end)
        self._opt_step += 1
        args = ops.AdamWArgs()
        sa, ta = self.s_arena, self.t_arena
        args.p, args.g, args.m, args.v = sa.fp32.data_ptr(), sa.grad.data_ptr(), sa.exp_avg.data_ptr(), sa.exp_avg_sq.data_ptr()
        args.p_bf16 = sa.bf16.data_ptr()
        if fuse_ema:
            args.t, args.t_bf16 = ta.fp32.data_ptr(), ta.bf16.data_ptr()
        args.n, args.chunk = sa.total, CHUNK
        args.lr_scale, args.wd_scale, args.flags = self.lr_table.data_ptr(), self.wd_table.data_ptr(), self.flag_table.data_ptr()
        args.lr, args.wd = lr, opt.weight_decay
        args.beta1, args.beta2, args.eps = self.optimizer_args.betas[0], self.optimizer_args.betas[1], self.optimizer_args.eps
        args.step, args.ema_m = self._opt_step, momentum
        args.gradnorm_sq = self.gradnorm_sq.data_ptr() if opt.clip_val is not None else None
        args.max_norm = float(opt.clip_val or 0.0)
        args.grad_scale = 1.0 / world
        args.freeze_last_layer = int(opt.freeze_last_layer)
        args.freeze_backbone = int(opt.freeze_backbone)
        ops.adamw_ema(args)
        sa.bf16_valid = True
        if fuse_ema:
            ta.bf16_valid = True
            self._ema_done = True
        self._grad_ready = False

    # ------------------------------------------------------------------ checkpoint (Lightning layout)
    def checkpoint(self) -> Dict[str, Any]:
        """{"state_dict", "optimizer_states", "lr_schedulers", "global_step"}: the keys of a Lightning checkpoint that
        this path owns.  `state_dict` carries the reference's parameter / buffer names (loads into the reference module)."""
        (opt,), (sch,) = self.configure_optimizers()
        return {"state_dict": {k: v.detach().clone() for k, v in self.state_dict().items()},
                "optimizer_states": [opt.state_dict()], "lr_schedulers": [sch["scheduler"].state_dict()],
                "global_step": self.trainer.global_step}

    def load_checkpoint(self, ckpt: Dict[str, Any]) -> None:
        (opt,), (sch,) = self.configure_optimizers()
        self.load_state_dict(ckpt["state_dict"])
        opt.load_state_dict(ckpt["optimizer_states"][0])
        sch["scheduler"].load_state_dict(ckpt["lr_schedulers"][0])
        self.trainer.global_step = int(ckpt["global_step"])

    @staticmethod
    def loss_for_autograd(result: TrainingStepResult) -> Tensor:
        """Bridge for trainers that call `loss.backward()` themselves (Lightning automatic optimisation): the
        gradients are already in `param.grad` when training_step_impl returns, so the returned leaf only has to
        make `backward()` a no-op instead of an error (INTEGRATION.md, 'autograd bridge')."""
        return result.loss.detach().requires_grad_(True)

    def release_graphs(self) -> None:
        """Drop the captured step graphs (and their memory pool).  Call before `dist.destroy_process_group()` when the graphs
        hold captured NCCL kernels (B200_GRAPH_NCCL=1): the communicator cannot be torn down while a graph references it."""
        st = self._static
        if st is not None:
            for entry in st["graphs"].values():
                for g in entry[:3]:
                    if g is not None:
                        g.reset()
            st["graphs"].clear()
            st["pool"] = None
        self._static = None

    def _graph_ok(self) -> bool:
        """CUDA-graph replay of the step.  With Sinkhorn-Knopp on several ranks the per-iteration [K] all-reduces sit in the
        middle of the captured schedule: they are captured into the graph (every rank then replays ONE padded shape every
        step, see `_graphed_step`), unless B200_GRAPH_NCCL=0, in which case that step runs eagerly."""
        if not self.use_cuda_graph:
            return False
        if self.method_args.center_method == "softmax" or _world_size() == 1:
            return True
        return GRAPH_NCCL

    def train_step(self, batch: Dict[str, Any]) -> TrainingStepResult:
        """One full optimisation step: what Lightning's fit loop does around training_step (SURVEY.md 3.1)."""
        ops._req_cuda(self.s_arena.fp32)
        if self._graph_ok():
            res = self._graphed_step(batch)
        else:
            res = self.training_step_impl(batch, 0)
        self.optimizer_step()
        return res


class FusedAdamWEMA:
    """Optimizer shim handed to the trainer by DINOv2.configure_optimizers: `step()` runs the fused sweep over the flat
    arenas.  `param_groups` mirror what get_optimizer_with_decay + get_fused_param_groups build (utils.py:191-273) so that
    hooks / loggers that read or edit lr / weight_decay by group name keep working; the sweep itself reads the per-chunk
    tables.  State (exp_avg, exp_avg_sq, step) round-trips through state_dict() like torch.optim.AdamW's."""

    def __init__(self, method: DINOv2) -> None:
        self.method = method
        self.clip_val: Optional[float] = None
        self.weight_decay = method.weight_decay_start
        self.freeze_backbone = False
        self.freeze_last_layer = False
        self.defaults = dict(lr=method.base_lr, betas=method.optimizer_args.betas, eps=method.optimizer_args.eps,
                             weight_decay=method.optimizer_args.weight_decay)
        groups: Dict[Tuple[float, float, bool, bool], Dict[str, Any]] = {}
        nl = method.s_vit.n_blocks
        a = method.method_args
        for full in method.s_arena.names():
            is_bb = full.startswith("backbone.")
            st = param_group_settings(full[len("backbone."):] if is_bb else full, is_bb, nl, a.layerwise_decay,
                                      a.patch_embed_lr_multiplier)
            key = (st["lr_scale"], st["wd_scale"], bool(st["last_layer"]), not is_bb)
            g = groups.get(key)
            if g is None:
                # reference group names: parameter names inside trainable_modules() (the ViT itself, then DINOv2Head)
                g = groups[key] = {"name": full[len("backbone."):] if is_bb else full, "params": [], "lr_scale": st["lr_scale"],
                                   "wd_scale": st["wd_scale"], "lr": method.base_lr * st["lr_scale"],
                                   "weight_decay": self.weight_decay * st["wd_scale"], "is_last_layer": bool(st["last_layer"]),
                                   "is_head": not is_bb}
            g["params"].append(method.s_arena.p(full))
        self.param_groups: List[Dict[str, Any]] = list(groups.values())

    def sync_param_groups(self, lr: Optional[float] = None) -> None:
        lr = self.method.base_lr * self.method._scheduler.factor() if lr is None else lr
        for g in self.param_groups:
            frozen = (self.freeze_last_layer and g["is_last_layer"]) or (self.freeze_backbone and not g["is_head"])
            g["lr"] = 0.0 if frozen else lr * g["lr_scale"]
            g["weight_decay"] = self.weight_decay * g["wd_scale"]

    def zero_grad(self, set_to_none: bool = False) -> None:
        """Gradients live in the flat arena and are zeroed by the step's first kernel."""

    def step(self, closure: Any = None) -> None:
        if closure is not None:
            closure()
        m = self.method
        if not m._grad_ready:
            raise RuntimeError("optimizer.step() without gradients; call training_step / training_step_impl first")
        m._fused_sweep(self, m.base_lr * m._scheduler.factor())

    def state_dict(self) -> Dict[str, Any]:
        sa = self.method.s_arena
        return {"exp_avg": sa.exp_avg.detach().clone(), "exp_avg_sq": sa.exp_avg_sq.detach().clone(),
                "step": self.method._opt_step,
                "param_groups": [{k: v for k, v in g.items() if k != "params"} for g in self.param_groups]}

    def load_state_dict(self, sd: Dict[str, Any]) -> None:
        sa = self.method.s_arena
        sa.exp_avg.copy_(sd["exp_avg"])
        sa.exp_avg_sq.copy_(sd["exp_avg_sq"])
        self.method._opt_step = int(sd["step"])


class CosineWarmupFactor:
    """lightly's CosineWarmupScheduler as the reference configures it (:576-583): `last_epoch` counts scheduler steps."""

    def __init__(self, method: DINOv2) -> None:
        self.method = method
        self.last_epoch = 0

    def factor(self) -> float:
        m = self.method
        max_steps = int(m.trainer.estimated_stepping_batches)
        warmup = int(min(max_steps - 1, m.method_args.warmup_steps))
        return cosine_warmup_factor(self.last_epoch, warmup, max_steps, m.method_args.min_lr / m.base_lr)

    def step(self) -> None:
        self.last_epoch += 1

    def get_last_lr(self) -> List[float]:
        f = self.factor()
        return [self.method.base_lr * f * g["lr_scale"] for g in self.method._optimizer.param_groups]

    def state_dict(self) -> Dict[str, Any]:
        return {"last_epoch": self.last_epoch}

    def load_state_dict(self, sd: Dict[str, Any]) -> None:
        self.last_epoch = int(sd["last_epoch"])
