"""Generate the method-level fixtures under tests/golden/ by running the reference's OWN method classes (DINOv2,
DistillationV3, DinoVisionTransformer; through oracle/ref_full.py) on the seeded weights and inputs of
tests/golden/recipes.py and tests/ref_cases.py.  Needs the reference source:

    LIGHTLY_TRAIN_SRC=<lightly-train checkout>/src python tools/make_method_golden.py

Whole gradients and weights would make the fixtures large: for every tensor they keep its norm and the elements at
`recipes.sample_index`, which the tests compare at the same positions.
"""
from __future__ import annotations

import dataclasses
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from oracle import ref_full  # noqa: E402
from tests import ref_cases as RC  # noqa: E402
from tests.golden import recipes as R  # noqa: E402

OUT = ROOT / "tests" / "golden"
SAMPLE = 32  # elements kept per tensor


def _ref_name(k: str) -> str:
    """oracle flat name of a student tensor -> reference method state_dict name."""
    if k.startswith("backbone."):
        return "student_embedding_model.wrapped_model._model." + k[len("backbone."):]
    return "student_head." + k


def _sampled(tensors: dict, names: list) -> torch.Tensor:
    return torch.stack([tensors[k].detach().float().flatten()[R.sample_index(tensors[k].numel(), SAMPLE)] for k in names])


def method_step_case(case: RC.Case) -> dict:
    """One optimisation step of the reference DINOv2 method (training_step_impl, backward, then its hooks in Lightning's
    order) from the recipe weights: loss terms, gradients and the student / teacher weights after the step."""
    m, opt, sched = RC.build_reference(case, max_steps=10)
    cfg = RC.oracle_cfg(case)
    st = R.det_step_state(cfg, seed=41)
    RC.load_oracle_state(m, st["student"], st["teacher"], st["centers"])
    views = RC.make_views(case)
    terms, grads = RC.reference_losses(m, views, mask_seed=11)
    m.on_before_optimizer_step(opt)
    m.configure_gradient_clipping(opt)
    opt.step()
    sched.step()
    m.trainer.global_step += 1
    m.on_train_batch_end(None, {"views": views}, 0)
    s_after, t_after, _ = RC.oracle_state(m.state_dict(), cfg.ibot_separate_head)
    names = list(st["student"])
    g = {k: grads[_ref_name(k)] for k in names}
    a = m.method_args
    return {"terms": terms, "names": names,
            "args": {k: float(getattr(a, k)) for k in ("gradient_clip_val", "min_lr", "weight_decay_end", "momentum_start", "momentum_end")},
            "grad_norm": torch.tensor([g[k].norm().item() for k in names]), "grad_sample": _sampled(g, names),
            "student_after": _sampled(s_after, names), "teacher_after": _sampled(t_after, names)}


def parity_case(case: RC.Case) -> dict:
    """Loss terms and gradients of the reference DINOv2 method in fp32 at a BASELINE.json configuration (KoLeo weight 0,
    as tests/test_parity_configs_gpu.py runs it), from the recipe weights."""
    torch.set_num_threads(32)
    case = dataclasses.replace(case, method=dict(case.method, koleo_loss_weight=0.0))
    cfg = dataclasses.replace(RC.oracle_cfg(case), koleo_loss_weight=0.0)
    m, _, _ = RC.build_reference(case)
    st = R.det_step_state(cfg, seed=41)
    RC.load_oracle_state(m, st["student"], st["teacher"], st["centers"])
    terms, grads = RC.reference_losses(m, RC.make_views(case), mask_seed=11)
    names = [k for k in st["student"] if _ref_name(k) in grads]
    g = {k: grads[_ref_name(k)] for k in names}
    return {"terms": terms, "names": names, "grad_norm": torch.tensor([g[k].norm().item() for k in names]),
            "grad_sample": _sampled(g, names)}


BOUNDARY_CASES = [
    (dict(img_size=224, patch_size=16, embed_dim=128, depth=4, num_heads=2, init_values=1e-5, drop_path_rate=0.3),
     dict(output_dim=512, hidden_dim=256)),
    (dict(img_size=224, patch_size=14, embed_dim=128, depth=2, num_heads=2, init_values=1e-5, drop_path_rate=0.2, drop_path_uniform=True,
          ffn_layer="swiglufused", num_register_tokens=4, interpolate_antialias=True, interpolate_offset=0.0),
     dict(output_dim=512, hidden_dim=256, ibot_separate_head=True, center_method="sinkhorn_knopp")),
]


def _layout(sd: dict) -> list:
    return [[k, list(v.shape)] for k, v in sd.items()]


def boundary_case() -> dict:
    """What the drop-in boundary tests compare with: state_dict layouts of the reference method and ViT, the attributes a
    pre-built reference backbone presents to a constructor, and the optimizer groups and per-step hook values."""
    ref_full.install()
    from lightly_train._models.dinov2_vit.dinov2_vit_src.models.vision_transformer import DinoVisionTransformer  # type: ignore
    out: dict = {"constructor": []}
    for vit_kw, method_kw in BOUNDARY_CASES:
        torch.manual_seed(0)
        ref, _, _ = ref_full.build_dinov2(dict(vit_kw, block_chunks=0), dict(method_kw), global_batch_size=64, max_steps=20)
        vit = DinoVisionTransformer(**dict(vit_kw, block_chunks=0))
        attrs = {k: getattr(vit, k) for k in ("embed_dim", "n_blocks", "num_heads", "patch_size", "num_register_tokens",
                                              "interpolate_antialias", "interpolate_offset", "chunked_blocks")}
        out["constructor"].append({"method_state_dict": _layout(ref.state_dict()), "backbone_attrs": attrs,
                                   "backbone_sample_drop_ratio": [float(getattr(b, "sample_drop_ratio", 0.0)) for b in vit.blocks],
                                   "backbone_state_dict": _layout(vit.state_dict())})
    vit_kw = dict(img_size=224, patch_size=16, embed_dim=128, depth=4, num_heads=2, init_values=1e-5, drop_path_rate=0.0)
    mk = dict(output_dim=512, hidden_dim=256, warmup_steps=3, student_freeze_last_layer_steps=2, student_freeze_backbone_steps=1)
    torch.manual_seed(0)
    ref, ropt, rsched = ref_full.build_dinov2(dict(vit_kw, block_chunks=0), mk, global_batch_size=64, max_steps=8)
    groups = [[g["name"], sum(p.numel() for p in g["params"])] for g in ropt.param_groups]
    lr, wd = [], []
    for _ in range(8):
        ref.on_before_optimizer_step(ropt)
        lr.append([g["lr"] for g in ropt.param_groups])
        wd.append([g["weight_decay"] for g in ropt.param_groups])
        ropt.step(); rsched.step(); ref.trainer.global_step += 1
    out["hooks"] = {"groups": groups, "lr": lr, "weight_decay": wd}
    r = DinoVisionTransformer(embed_dim=128, depth=4, num_heads=2, block_chunks=2, init_values=1e-5)
    out["chunked_vit_state_dict"] = _layout(r.state_dict())
    out["tiny_method_state_dict"] = _layout(RC.build_reference(RC.TINY)[0].state_dict())
    return out


def distillation_case() -> dict:
    """Two training_step_impl calls of the reference DistillationV3 (DINOv3 ViT teacher, ResNet-18 student) on the recipe
    teacher / head weights: loss terms, the teacher queue, and gradients after the second step."""
    import torchvision

    ref_full.install()
    from lightly_train._methods.distillationv3.distillationv3 import DistillationV3 as RefMethod  # type: ignore
    from lightly_train._methods.distillationv3.distillationv3 import DistillationV3AdamWArgs, DistillationV3Args as RefArgs  # type: ignore
    from lightly_train._models.dinov3.dinov3_src.models import vision_transformer as v3  # type: ignore
    from lightly_train._models.dinov3.dinov3_vit import DINOv3ViTModelWrapper as RefTeacherWrapper  # type: ignore
    from lightly_train._models.embedding_model import EmbeddingModel as RefEmbedding  # type: ignore
    from lightly_train._models.torchvision.resnet import ResNetModelWrapper as RefResNetWrapper  # type: ignore

    rvit = v3.DinoVisionTransformer(**R.DISTILL_TEACHER_KW)
    rvit.init_weights()  # fills rope periods and the k-bias mask
    r = rvit.load_state_dict(R.det_dinov3_state(R.dinov3_tiny_cfg(), seed=15), strict=False)
    assert not r.unexpected_keys and all(k.endswith("bias_mask") or k == "rope_embed.periods" for k in r.missing_keys), r
    torch.manual_seed(0)
    resnet = torchvision.models.resnet18()
    rm = RefMethod(RefArgs(queue_size=64, teacher=RefTeacherWrapper(rvit)), DistillationV3AdamWArgs(),
                   RefEmbedding(wrapped_model=RefResNetWrapper(resnet)), global_batch_size=4, num_input_channels=3)
    rm.trainer = ref_full._Trainer(10)
    for n in ("student_projection_head_global", "student_projection_head_local"):
        R.det_fill_(getattr(rm, n), seed=16)
    x = R.distill_step_input()
    out: dict = {"steps": []}
    for step in range(2):  # second step: the queue already holds the first batch
        torch.manual_seed(100 + step)
        rres = rm.training_step_impl({"views": [x]}, 0)
        rows = 4 * (step + 1)
        assert not rm.teacher_queue[rows:].any()
        out["steps"].append({"global_loss": float(rres.log_dict["train_loss/global_loss"]),
                             "local_loss": float(rres.log_dict["train_loss/local_loss"]),
                             "queue_head": rm.teacher_queue[:rows].clone()})
    rres.loss.backward()
    res = rm.student_embedding_model.wrapped_model.get_model()
    g = {"head_global": rm.student_projection_head_global.weight.grad, "layer4.1.conv2": res.layer4[1].conv2.weight.grad,
         "conv1": res.conv1.weight.grad}
    out["grads"] = {k: {"norm": v.norm().item(), "sample": v.flatten()[R.sample_index(v.numel(), 2048)].clone()} for k, v in g.items()}
    return out


def main() -> None:
    if not ref_full.available():
        raise SystemExit("set LIGHTLY_TRAIN_SRC to the src directory of a lightly-train checkout")
    torch.set_num_threads(8)
    for case in (RC.TINY, RC.TINY_SK):
        torch.save(method_step_case(case), OUT / f"method_step_{case.name}.pt")
    for case in (RC.CFG1, RC.CFG2, RC.CFG3, RC.CFG5):
        torch.save(parity_case(case), OUT / f"parity_{case.name.split('_')[0]}.pt")
    (OUT / "method_boundary.json").write_text(json.dumps(boundary_case()))
    torch.save(distillation_case(), OUT / "distillation_v3_step.pt")
    for f in sorted(OUT.glob("*")):
        print(f.name, f.stat().st_size)


if __name__ == "__main__":
    main()
