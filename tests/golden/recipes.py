"""Deterministic recipes for the golden fixtures: configs, weights and inputs are regenerated from seeds
(torch CPU generator) so only the reference's OUTPUTS need to be stored under tests/golden/.

Weights deliberately use O(1) LayerScale gammas and non-trivial norms/biases: the reference initialisation
(gamma=1e-5, zero biases) makes every block a near-identity and would hide kernel errors.
"""
from __future__ import annotations

from typing import Dict, List, Tuple

import torch
from torch import Tensor

from oracle import dinov2_oracle as O

VIT_TINY = O.ViTConfig(embed_dim=128, depth=2, num_heads=2, patch_size=16, img_size=224, init_values=1e-5)
VIT_TINY_REG = O.ViTConfig(embed_dim=128, depth=2, num_heads=2, patch_size=16, img_size=224, init_values=1e-5,
                           num_register_tokens=4, interpolate_offset=0.0, interpolate_antialias=True)
VIT_TINY_SWIGLU = O.ViTConfig(embed_dim=128, depth=2, num_heads=2, patch_size=16, img_size=224, init_values=1e-5,
                              num_register_tokens=4, ffn_layer="swiglu")  # cfg3's zoo default FFN (hidden 344)
HEAD_TINY = O.HeadConfig(in_dim=128, hidden_dim=256, bottleneck_dim=64, out_dim=512)


def vit_param_shapes(cfg: O.ViTConfig) -> Dict[str, Tuple[int, ...]]:
    D, H, p = cfg.embed_dim, cfg.hidden_dim, cfg.patch_size
    shapes: Dict[str, Tuple[int, ...]] = {
        "cls_token": (1, 1, D), "pos_embed": (1, 1 + cfg.num_patches, D), "mask_token": (1, D),
        "patch_embed.proj.weight": (D, 3, p, p), "patch_embed.proj.bias": (D,),
    }
    if cfg.num_register_tokens:
        shapes["register_tokens"] = (1, cfg.num_register_tokens, D)
    for i in range(cfg.depth):
        b = f"blocks.{i}."
        shapes.update({
            b + "norm1.weight": (D,), b + "norm1.bias": (D,),
            b + "attn.qkv.weight": (3 * D, D), b + "attn.qkv.bias": (3 * D,),
            b + "attn.proj.weight": (D, D), b + "attn.proj.bias": (D,),
            b + "ls1.gamma": (D,),
            b + "norm2.weight": (D,), b + "norm2.bias": (D,),
        })
        if cfg.ffn_layer == "mlp":
            shapes.update({b + "mlp.fc1.weight": (H, D), b + "mlp.fc1.bias": (H,),
                           b + "mlp.fc2.weight": (D, H), b + "mlp.fc2.bias": (D,)})
        else:
            shapes.update({b + "mlp.w12.weight": (2 * H, D), b + "mlp.w12.bias": (2 * H,),
                           b + "mlp.w3.weight": (D, H), b + "mlp.w3.bias": (D,)})
        shapes.update({
            b + "ls2.gamma": (D,),
        })
    shapes.update({"norm.weight": (D,), "norm.bias": (D,)})
    return shapes


def head_param_shapes(cfg: O.HeadConfig) -> Dict[str, Tuple[int, ...]]:
    return {
        "mlp.0.weight": (cfg.hidden_dim, cfg.in_dim), "mlp.0.bias": (cfg.hidden_dim,),
        "mlp.2.weight": (cfg.hidden_dim, cfg.hidden_dim), "mlp.2.bias": (cfg.hidden_dim,),
        "mlp.4.weight": (cfg.bottleneck_dim, cfg.hidden_dim), "mlp.4.bias": (cfg.bottleneck_dim,),
        "last_layer.parametrizations.weight.original0": (cfg.out_dim, 1),
        "last_layer.parametrizations.weight.original1": (cfg.out_dim, cfg.bottleneck_dim),
    }


def _fill(name: str, shape: Tuple[int, ...], g: torch.Generator) -> Tensor:
    r = torch.randn(shape, generator=g)
    if name.endswith("norm1.weight") or name.endswith("norm2.weight") or name == "norm.weight":
        return 1.0 + 0.1 * r
    if "gamma" in name:
        return 0.5 + 0.1 * r
    if name.endswith("original0"):
        return 1.0 + 0.05 * r
    if name.endswith(".bias"):
        return 0.05 * r
    if name in ("cls_token", "mask_token", "register_tokens"):
        return 0.1 * r
    if name == "pos_embed":
        return 0.1 * r
    if name == "patch_embed.proj.weight":
        return 0.03 * r
    if name.endswith("original1"):
        return 0.1 * r
    fan_in = shape[-1]
    return r * (0.7 / fan_in ** 0.5)


def sample_index(numel: int, n: int) -> Tensor:
    """n distinct flat indices spread over a tensor of `numel` elements (all of them when numel <= n): where a fixture
    would otherwise hold a whole gradient or weight tensor, it holds these elements only."""
    if numel <= n:
        return torch.arange(numel)
    return (torch.arange(n, dtype=torch.int64) * 2654435761 + 97) % numel  # prime stride: distinct for numel < 2654435761


def det_vit_state(cfg: O.ViTConfig, seed: int) -> Dict[str, Tensor]:
    g = torch.Generator().manual_seed(seed)
    return {k: _fill(k, s, g) for k, s in vit_param_shapes(cfg).items()}


def det_head_state(cfg: O.HeadConfig, seed: int) -> Dict[str, Tensor]:
    g = torch.Generator().manual_seed(seed)
    return {k: _fill(k, s, g) for k, s in head_param_shapes(cfg).items()}


def vit_case_inputs() -> Tuple[Tensor, Tensor, Tensor]:
    g = torch.Generator().manual_seed(101)
    xg = torch.randn(2, 3, 224, 224, generator=g)
    xl = torch.randn(3, 3, 96, 96, generator=g)
    masks = torch.rand(2, 196, generator=g) < 0.3
    masks[1] = False
    return xg, xl, masks


def vit_swiglu_cotangents() -> Tuple[Tensor, Tensor]:
    g = torch.Generator().manual_seed(104)
    return torch.randn(2, 196, VIT_TINY_SWIGLU.embed_dim, generator=g), torch.randn(2, VIT_TINY_SWIGLU.embed_dim, generator=g)


def head_case_input() -> Tensor:
    g = torch.Generator().manual_seed(102)
    return torch.randn(37, HEAD_TINY.in_dim, generator=g)


def head_case_cotangent() -> Tensor:
    g = torch.Generator().manual_seed(103)
    return torch.randn(37, HEAD_TINY.out_dim, generator=g) * 0.1


def step_config(center_method: str, separate: bool) -> O.StepConfig:
    return O.StepConfig(vit=VIT_TINY, head=HEAD_TINY, ibot_separate_head=separate, center_method=center_method)


def det_step_state(cfg: O.StepConfig, seed: int) -> Dict[str, Dict[str, Tensor]]:
    """student/teacher flat dicts ("backbone.", "dino_head.", "ibot_head." prefixes) + loss centers."""
    out: Dict[str, Dict[str, Tensor]] = {}
    for j, who in enumerate(("student", "teacher")):
        sd: Dict[str, Tensor] = {}
        for k, v in det_vit_state(cfg.vit, seed + 10 * j).items():
            sd["backbone." + k] = v
        for k, v in det_head_state(cfg.head, seed + 10 * j + 1).items():
            sd["dino_head." + k] = v
        if cfg.ibot_separate_head:
            for k, v in det_head_state(cfg.head, seed + 10 * j + 2).items():
                sd["ibot_head." + k] = v
        out[who] = sd
    g = torch.Generator().manual_seed(seed + 99)
    K = cfg.head.out_dim
    out["centers"] = {"dino": 0.1 * torch.randn(1, K, generator=g), "ibot": 0.1 * torch.randn(1, 1, K, generator=g)}
    return out


def step_case_inputs(cfg: O.StepConfig, batch: int = 3, n_local: int = 2) -> Tuple[List[Tensor], Tensor, Tensor, Tensor]:
    g = torch.Generator().manual_seed(104)
    views = [torch.randn(batch, 3, 224, 224, generator=g) for _ in range(2)]
    views += [torch.randn(batch, 3, 96, 96, generator=g) for _ in range(n_local)]
    masks = torch.rand(2 * batch, cfg.vit.num_patches, generator=g) < 0.25
    masks[1] = False
    masks[4] = False
    idx = masks.flatten().nonzero().flatten()
    w = O.masks_weight_from_masks(masks)
    return views, masks, idx, w


def distill_case_inputs():
    """(teacher_global, teacher_local, student_global, student_local, queue), all L2-normalised; B=4, M=9 tokens, D=16, C=32."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(301)
    B, M, D, C = 4, 9, 16, 32
    tg = F.normalize(torch.randn(B, D, generator=g), dim=-1)
    tl = F.normalize(torch.randn(B, M, D, generator=g), dim=-1)
    sg = F.normalize(torch.randn(B, D, generator=g), dim=-1)
    sl = F.normalize(torch.randn(B, M, D, generator=g), dim=-1)
    q = F.normalize(torch.randn(C, D, generator=g), dim=-1)
    return tg, tl, sg, sl, q


# ---------------------------------------------------------------- DINOv3 teacher forward (distillation, SURVEY 8a row a17)
def dinov3_tiny_cfg():
    from oracle import dinov3_oracle as D3
    return D3.Dinov3Config(embed_dim=128, depth=2, num_heads=2, patch_size=16)


def dinov3_param_shapes(cfg) -> Dict[str, Tuple[int, ...]]:
    D, p, H = cfg.embed_dim, cfg.patch_size, int(cfg.embed_dim * cfg.ffn_ratio)
    shapes: Dict[str, Tuple[int, ...]] = {
        "cls_token": (1, 1, D), "storage_tokens": (1, cfg.n_storage_tokens, D), "mask_token": (1, D),
        "patch_embed.proj.weight": (D, 3, p, p), "patch_embed.proj.bias": (D,),
    }
    for i in range(cfg.depth):
        b = f"blocks.{i}."
        shapes.update({
            b + "norm1.weight": (D,), b + "norm1.bias": (D,),
            b + "attn.qkv.weight": (3 * D, D), b + "attn.qkv.bias": (3 * D,),
            b + "attn.proj.weight": (D, D), b + "attn.proj.bias": (D,),
            b + "ls1.gamma": (D,),
            b + "norm2.weight": (D,), b + "norm2.bias": (D,),
            b + "mlp.fc1.weight": (H, D), b + "mlp.fc1.bias": (H,),
            b + "mlp.fc2.weight": (D, H), b + "mlp.fc2.bias": (D,),
            b + "ls2.gamma": (D,),
        })
    shapes.update({"norm.weight": (D,), "norm.bias": (D,)})
    return shapes


def det_dinov3_state(cfg, seed: int) -> Dict[str, Tensor]:
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k, shp in dinov3_param_shapes(cfg).items():
        out[k] = _fill("register_tokens" if k == "storage_tokens" else k, shp, g)
    return out


# ---------------------------------------------------------------- DistillationV3 step (DINOv3 teacher -> ResNet-18 student)
DISTILL_TEACHER_KW = dict(img_size=224, patch_size=16, embed_dim=128, depth=2, num_heads=2, ffn_ratio=4.0, layerscale_init=1e-5,
                          norm_layer="layernormbf16", n_storage_tokens=4, mask_k_bias=True, pos_embed_rope_dtype="fp32")


def det_fill_(module: torch.nn.Module, seed: int) -> None:
    """Deterministic weights for a module whose parameter names are the same on both sides (biases small, matrices
    0.7 / sqrt(fan_in))."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for k, p in sorted(module.named_parameters()):
            p.copy_(_fill(k, tuple(p.shape), g))


def distill_step_input() -> Tensor:
    return torch.randn(4, 3, 224, 224, generator=torch.Generator().manual_seed(403))


def dinov3_case_inputs() -> Tuple[Tensor, Tensor]:
    """Non-square image (14 x 6 patches) so that the axial RoPE's row / column roles are pinned, 30 % masked."""
    g = torch.Generator().manual_seed(402)
    x = torch.randn(2, 3, 224, 96, generator=g)
    masks = torch.rand(2, 14 * 6, generator=g) < 0.3
    return x, masks
