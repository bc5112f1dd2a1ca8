"""BASELINE.json configurations as parity cases, and helpers that drive the reference's OWN method class (through
oracle/ref_full.py: reference source from $LIGHTLY_TRAIN_SRC or baseline/_ref, absent third-party packages stubbed) next
to the oracle and the CUDA mirror on identical weights, crops and masks.  The tests compare with what
tools/make_method_golden.py stored from such runs under tests/golden/; only that tool needs the reference."""
from __future__ import annotations

import random
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional, Tuple

import torch
from torch import Tensor

from oracle import dinov2_oracle as O
from oracle import ref_full


@dataclass
class Case:
    name: str
    vit: Dict[str, Any]                       # DinoVisionTransformer kwargs (reference spelling)
    method: Dict[str, Any] = field(default_factory=dict)   # DINOv2Args overrides
    batch: int = 4
    n_local: int = 8
    local_size: int = 96
    global_size: int = 224
    checkpointing: bool = False
    seed: int = 0


def _vit(embed_dim, depth, heads, patch=16, **kw):
    d = dict(img_size=224, patch_size=patch, embed_dim=embed_dim, depth=depth, num_heads=heads, mlp_ratio=4, init_values=1e-5,
             drop_path_rate=0.0, block_chunks=0)
    d.update(kw)
    return d


# BASELINE.json `configs` at their real model dimensions (batch reduced: the CPU reference/oracle run in seconds)
CFG1 = Case("cfg1_vitt16_globals_only_bs4", _vit(192, 12, 3), batch=4, n_local=0)
CFG2 = Case("cfg2_vits16_2g8l_K65536", _vit(384, 12, 6), batch=4, n_local=8)
CFG3 = Case("cfg3_vitb14_reg4_swiglu_ibot_sinkhorn",
            _vit(768, 12, 12, patch=14, ffn_layer="swiglufused", num_register_tokens=4, interpolate_antialias=True,
                 interpolate_offset=0.0),
            method=dict(ibot_separate_head=True, center_method="sinkhorn_knopp"), batch=2, n_local=2, local_size=98)
CFG5 = Case("cfg5_vitl16_2g10l_ckpt", _vit(1024, 24, 16), batch=2, n_local=10, checkpointing=True)
TINY = Case("tiny", _vit(128, 2, 2), method=dict(output_dim=512, hidden_dim=256, dino_bottleneck_dim=64, ibot_bottleneck_dim=64),
            batch=3, n_local=2)
TINY_SK = Case("tiny_sinkhorn_sep", _vit(128, 2, 2),
               method=dict(output_dim=512, hidden_dim=256, dino_bottleneck_dim=64, ibot_bottleneck_dim=64,
                           ibot_separate_head=True, center_method="sinkhorn_knopp"), batch=3, n_local=2)


def make_views(case: Case, seed: int = 0) -> List[Tensor]:
    g = torch.Generator().manual_seed(1234 + seed)
    v = [torch.randn(case.batch, 3, case.global_size, case.global_size, generator=g) for _ in range(2)]
    v += [torch.randn(case.batch, 3, case.local_size, case.local_size, generator=g) for _ in range(case.n_local)]
    return v


def perturb_(module: torch.nn.Module, seed: int) -> None:
    """The reference initialisation (LayerScale 1e-5, zero biases, unit norms) makes every block a near-identity and
    hides kernel errors: give gammas / biases / norm weights O(1) deterministic values (both sides get the same ones
    because the mirror loads the reference's state_dict afterwards)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in module.named_parameters():
            r = torch.randn(p.shape, generator=g)
            if n.endswith("gamma"):
                p.copy_(0.5 + 0.1 * r)
            elif "norm" in n and n.endswith("weight"):
                p.copy_(1.0 + 0.1 * r)
            elif n.endswith("bias"):
                p.copy_(0.05 * r)
            elif n.endswith(("cls_token", "mask_token", "register_tokens")):
                p.copy_(0.1 * r)
            elif n.endswith("original0"):
                p.copy_(1.0 + 0.05 * r)


def build_reference(case: Case, max_steps: int = 100, device: str = "cpu", global_batch_size: Optional[int] = None):
    torch.manual_seed(case.seed)
    margs = dict(warmup_steps=2, student_freeze_last_layer_steps=1, teacher_temp_start=0.05, teacher_temp_end=0.05)
    margs.update(case.method)
    m, opt, sched = ref_full.build_dinov2(case.vit, margs, global_batch_size or case.batch, max_steps, device="cpu")
    perturb_(m.student_embedding_model, 1)
    perturb_(m.student_head, 2)
    perturb_(m.teacher_embedding_model, 3)
    perturb_(m.teacher_head, 4)
    with torch.no_grad():
        g = torch.Generator().manual_seed(5)
        m.dino_loss.center.copy_(0.1 * torch.randn(m.dino_loss.center.shape, generator=g))
        m.ibot_loss.center.copy_(0.1 * torch.randn(m.ibot_loss.center.shape, generator=g))
    if case.checkpointing:
        m.student_embedding_model.wrapped_model.set_activation_checkpointing(True)
    if device != "cpu":
        m.to(device)
    return m, opt, sched


def oracle_state(ref_state: Dict[str, Tensor], separate: bool) -> Tuple[Dict[str, Tensor], Dict[str, Tensor], Dict[str, Tensor]]:
    """reference method state_dict -> (student, teacher, centers) in the oracle's flat naming."""
    out = {"student": {}, "teacher": {}}
    for who in ("student", "teacher"):
        bb = f"{who}_embedding_model.wrapped_model._model."
        for k, v in ref_state.items():
            if k.startswith(bb):
                out[who]["backbone." + k[len(bb):]] = v.detach().clone().float()
            elif k.startswith(f"{who}_head.dino_head."):
                out[who]["dino_head." + k[len(f"{who}_head.dino_head."):]] = v.detach().clone().float()
            elif separate and k.startswith(f"{who}_head.ibot_head."):
                out[who]["ibot_head." + k[len(f"{who}_head.ibot_head."):]] = v.detach().clone().float()
    centers = {"dino": ref_state["dino_loss.center"].clone(), "ibot": ref_state["ibot_loss.center"].clone()}
    return out["student"], out["teacher"], centers


def load_oracle_state(m, student: Dict[str, Tensor], teacher: Dict[str, Tensor], centers: Dict[str, Tensor]) -> None:
    """Inverse of `oracle_state`: write flat oracle weights into a method's state_dict (reference or mirror naming); a
    shared iBOT head takes the DINO head's weights."""
    sd = m.state_dict()
    new = {}
    for who, flat in (("student", student), ("teacher", teacher)):
        for k, v in flat.items():
            if k.startswith("backbone."):
                new[f"{who}_embedding_model.wrapped_model._model." + k[len("backbone."):]] = v
            else:
                new[f"{who}_head." + k] = v
                if k.startswith("dino_head.") and f"{who}_head.ibot_{k[len('dino_'):]}" in sd and "ibot_head." + k[len("dino_head."):] not in flat:
                    new[f"{who}_head.ibot_{k[len('dino_'):]}"] = v
    new["dino_loss.center"], new["ibot_loss.center"] = centers["dino"], centers["ibot"]
    assert set(new) == set(sd), set(new) ^ set(sd)
    m.load_state_dict({k: new[k].reshape(sd[k].shape) for k in sd}, strict=True)


def oracle_cfg(case: Case) -> O.StepConfig:
    v = case.vit
    vit = O.ViTConfig(embed_dim=v["embed_dim"], depth=v["depth"], num_heads=v["num_heads"], patch_size=v["patch_size"],
                      img_size=v["img_size"], init_values=v["init_values"], num_register_tokens=v.get("num_register_tokens", 0),
                      interpolate_offset=v.get("interpolate_offset", 0.1), interpolate_antialias=v.get("interpolate_antialias", False),
                      ffn_layer=v.get("ffn_layer", "mlp"))
    m = case.method
    head = O.HeadConfig(in_dim=v["embed_dim"], hidden_dim=m.get("hidden_dim", 2048), bottleneck_dim=m.get("dino_bottleneck_dim", 256),
                        out_dim=m.get("output_dim", 65536))
    return O.StepConfig(vit=vit, head=head, ibot_separate_head=m.get("ibot_separate_head", False),
                        center_method=m.get("center_method", "softmax"))


def masks_for(case: Case, mask_seed: int) -> Dict[str, Tensor]:
    """The masks the reference's training_step_impl draws from python `random` after random.seed(mask_seed), produced by
    the mirror's bit-exact generator (tests/test_host_logic.py pins it against the reference's own)."""
    from lightly_train_b200._methods.dinov2.utils import MaskingGenerator, create_collated_masks
    p = case.vit["patch_size"]
    h = w = case.global_size // p
    random.seed(mask_seed)
    gen = MaskingGenerator(input_size=(h, w), max_num_patches=int(0.5 * h * w))
    return create_collated_masks(0.1, 0.5, int(2 * case.batch * 0.5), 2 * case.batch, gen)


def reference_losses(m, views: List[Tensor], mask_seed: int, autocast_device: Optional[str] = None):
    """Forward + backward of the reference method's own training_step_impl; returns (loss terms, grads by state_dict name)."""
    random.seed(mask_seed)
    for p in m.parameters():
        p.grad = None
    if autocast_device:
        with torch.autocast(autocast_device, dtype=torch.bfloat16):
            res = m.training_step_impl({"views": views}, 0)
    else:
        res = m.training_step_impl({"views": views}, 0)
    res.loss.backward()
    terms = {"loss": float(res.loss)}
    terms.update({k.split("/")[1]: float(v) for k, v in res.log_dict.items()})
    grads = {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}
    return terms, grads
