"""CPU: the drop-in boundary against the reference's OWN method class without touching a GPU: reference constructor
(pre-built embedding model), state_dict names / shapes both ways, optimizer param groups, and the per-step lr /
weight-decay / freeze values the hooks produce (dinov2.py:550-639).  What the reference presents and produces was stored
by tools/make_method_golden.py (through oracle/ref_full.py) in tests/golden/method_boundary.json."""
import json

import pytest
import torch
from torch import nn

VIT_CASES = [
    (dict(img_size=224, patch_size=16, embed_dim=128, depth=4, num_heads=2, init_values=1e-5, drop_path_rate=0.3), dict(output_dim=512, hidden_dim=256)),
    (dict(img_size=224, patch_size=14, embed_dim=128, depth=2, num_heads=2, init_values=1e-5, drop_path_rate=0.2, drop_path_uniform=True,
          ffn_layer="swiglufused", num_register_tokens=4, interpolate_antialias=True, interpolate_offset=0.0),
     dict(output_dim=512, hidden_dim=256, ibot_separate_head=True, center_method="sinkhorn_knopp")),
]


@pytest.fixture(scope="module")
def boundary(golden_dir):
    return json.loads((golden_dir / "method_boundary.json").read_text())


class _Wrapper:
    """EmbeddingModel(wrapped_model=DINOv2ViTModelWrapper(vit)) as the reference spells it."""

    def __init__(self, vit: nn.Module) -> None:
        self.wrapped_model = self
        self._vit = vit

    def get_model(self) -> nn.Module:
        return self._vit


def _reference_backbone(desc: dict) -> nn.Module:
    """A module with the parameter names / shapes, block list and attributes of the reference DinoVisionTransformer the
    fixture describes, seeded random weights: what a caller hands to the constructor."""
    g = torch.Generator().manual_seed(7)
    vit = nn.Module()
    vit.blocks = nn.ModuleList(nn.Module() for _ in desc["backbone_sample_drop_ratio"])
    for blk, r in zip(vit.blocks, desc["backbone_sample_drop_ratio"]):
        blk.sample_drop_ratio = r
    for name, shape in desc["backbone_state_dict"]:
        *path, leaf = name.split(".")
        mod = vit
        for part in path:
            if part.isdigit():
                mod = mod[int(part)]
            else:
                if not hasattr(mod, part):
                    mod.add_module(part, nn.Module())
                mod = getattr(mod, part)
        mod.register_parameter(leaf, nn.Parameter(0.02 * torch.randn(shape, generator=g)))
    for k, v in desc["backbone_attrs"].items():
        setattr(vit, k, v)
    return vit


@pytest.mark.parametrize("vit_kw,method_kw", VIT_CASES)
def test_reference_constructor_and_state_dict(boundary, vit_kw, method_kw):
    from lightly_train_b200._methods.dinov2.dinov2 import DINOv2, DINOv2AdamWViTArgs, DINOv2Args
    desc = boundary["constructor"][VIT_CASES.index((vit_kw, method_kw))]
    # a FRESH reference backbone (with its stochastic depth) is what a caller hands to the constructor
    emb = _Wrapper(_reference_backbone(desc))
    mine = DINOv2(DINOv2Args(**method_kw), DINOv2AdamWViTArgs(), emb, 64, 3, max_steps=20, device="cpu")
    b = mine.state_dict()
    assert [[k, list(v.shape)] for k, v in b.items()] == desc["method_state_dict"]   # same names, same ORDER, same shapes
    # architecture read back from the module, incl. the stochastic-depth schedule of the student (teacher: none)
    s = mine.s_vit
    want = [float(x) for x in ([vit_kw["drop_path_rate"]] * vit_kw["depth"] if vit_kw.get("drop_path_uniform")
                               else torch.linspace(0, vit_kw["drop_path_rate"], vit_kw["depth"]).tolist())]
    assert s.dpr == pytest.approx(want) and mine.t_vit.dpr == [0.0] * vit_kw["depth"]
    assert s.swiglu == ("ffn_layer" in vit_kw) and s.num_register_tokens == vit_kw.get("num_register_tokens", 0)
    # the passed backbone's weights initialise BOTH sides (reference: student = deepcopy(teacher), dinov2.py:197-198)
    w = emb.wrapped_model.get_model().state_dict()["blocks.1.attn.qkv.weight"]
    assert torch.equal(b["teacher_embedding_model.wrapped_model._model.blocks.1.attn.qkv.weight"], w)
    assert torch.equal(b["student_embedding_model.wrapped_model._model.blocks.1.attn.qkv.weight"], w)
    # checkpoints flow both ways: a reference checkpoint loads strictly, and this one has the reference's exact layout
    g = torch.Generator().manual_seed(8)
    a = {k: torch.randn(shape, generator=g) for k, shape in desc["method_state_dict"]}
    res = mine.load_state_dict(a, strict=True)
    assert not res.missing_keys and not res.unexpected_keys


def test_param_groups_and_hook_schedules_match_reference(boundary):
    """Same group names, lr multipliers and weight-decay switches as get_optimizer_with_decay + get_fused_param_groups, and the
    same per-step lr (warm-up + cosine), weight decay (cosine) and freeze decisions as the reference's hooks, step by step."""
    from lightly_train_b200._methods.dinov2.dinov2 import DINOv2, DINOv2AdamWViTArgs, DINOv2Args
    vit_kw = dict(img_size=224, patch_size=16, embed_dim=128, depth=4, num_heads=2, init_values=1e-5, drop_path_rate=0.0)
    mk = dict(output_dim=512, hidden_dim=256, warmup_steps=3, student_freeze_last_layer_steps=2, student_freeze_backbone_steps=1)
    torch.manual_seed(0)
    mine = DINOv2(DINOv2Args(**mk), DINOv2AdamWViTArgs(), vit_kw, 64, 3, max_steps=8, device="cpu")
    ref = boundary["hooks"]
    (opt,), (sch,) = mine.configure_optimizers()
    mg = {g["name"]: g for g in opt.param_groups}
    assert [n for n, _ in ref["groups"]] == list(mg)
    assert all(sum(p.numel() for p in mg[n]["params"]) == numel for n, numel in ref["groups"])
    for step in range(8):
        mine.on_before_optimizer_step(opt)
        for j, (n, _) in enumerate(ref["groups"]):
            assert mg[n]["lr"] == pytest.approx(ref["lr"][step][j], rel=1e-6, abs=1e-12), (step, n)
            assert mg[n]["weight_decay"] == pytest.approx(ref["weight_decay"][step][j], rel=1e-6), (step, n)
        assert opt.freeze_backbone == (step < 1) and opt.freeze_last_layer == (step < 2)
        # (no optimizer.step(): the schedules only depend on the counters)
        sch["scheduler"].step(); mine.trainer.global_step += 1
