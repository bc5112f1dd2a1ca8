"""CPU tests of the host-side mirror of the reference interface (no GPU, no kernels)."""
import random

import pytest
import torch
import torch.nn.functional as F

from lightly_train_b200._methods.dinov2 import scheduler, utils
from lightly_train_b200._models.pos_embed import pos_embed_operator
from oracle import dinov2_oracle as O


def test_masks_reproduce_reference_bit_for_bit(golden_dir):
    ref = torch.load(golden_dir / "masks.pt")
    for case in ref.values():
        random.seed(case["seed"])
        hw = case["hw"]
        gen = utils.MaskingGenerator(input_size=(hw, hw), max_num_patches=int(0.5 * hw * hw))
        got = utils.create_collated_masks(0.1, 0.5, int(case["n_crops"] * 0.5), case["n_crops"], gen)
        assert torch.equal(got["collated_masks"], case["collated_masks"])
        assert torch.equal(got["mask_indices_list"], case["mask_indices_list"])
        assert torch.equal(got["masks_weight"], case["masks_weight"])


def test_mask_generator_invariants():
    """tests/_methods/dinov2/test_utils.py style invariants."""
    random.seed(0)
    gen = utils.MaskingGenerator(input_size=(14, 14), max_num_patches=98)
    for n in (0, 4, 20, 60, 98):
        m = gen(n)
        assert m.shape == (14, 14) and m.dtype == bool and m.sum() <= max(n, 0)
    res = utils.create_collated_masks(0.1, 0.5, 4, 8, gen)
    assert res["collated_masks"].shape == (8, 196)
    assert res["mask_indices_list"].numel() == int(res["collated_masks"].sum())
    per_img = res["collated_masks"].sum(-1)
    assert (per_img == 0).sum() >= 4


def test_lr_decay_and_groups_follow_reference_rules():
    """get_vit_lr_decay_rate / get_optimizer_with_decay (utils.py:155-250) vs the oracle restatement."""
    names = ["cls_token", "pos_embed", "mask_token", "patch_embed.proj.weight", "patch_embed.proj.bias",
             "blocks.0.norm1.weight", "blocks.3.attn.qkv.weight", "blocks.11.mlp.fc2.bias", "blocks.5.ls1.gamma",
             "norm.weight", "norm.bias"]
    for n in names:
        s = utils.param_group_settings(n, True, 12, 0.9, 0.2)
        o = O.param_hparams(n, True, 1.0, 1.0, 12, 0.9, 0.2)
        assert s["lr_scale"] == pytest.approx(o["lr"]) and s["wd_scale"] == pytest.approx(o["weight_decay"])
    assert utils.param_group_settings("blocks.0.attn.qkv.weight", True, 12, 0.9, 0.2)["lr_scale"] == pytest.approx(0.9 ** 12)
    assert utils.param_group_settings("patch_embed.proj.weight", True, 12, 0.9, 0.2)["lr_scale"] == pytest.approx(0.2 * 0.9 ** 13)
    assert utils.param_group_settings("norm.weight", True, 12, 0.9, 0.2)["lr_scale"] == pytest.approx(1.0)
    h = utils.param_group_settings("dino_head.last_layer.parametrizations.weight.original1", False, 12, 0.9, 0.2)
    assert h["lr_scale"] == 1.0 and h["wd_scale"] == 1.0 and h["last_layer"] == 1.0 and h["head"] == 1.0
    assert utils.param_group_settings("dino_head.mlp.0.bias", False, 12, 0.9, 0.2)["wd_scale"] == 0.0


def test_schedules():
    assert scheduler.linear_warmup_schedule(0, 37500, 0.04, 0.07) == 0.04
    assert scheduler.linear_warmup_schedule(37500, 37500, 0.04, 0.07) == 0.07
    with pytest.raises(ValueError):
        scheduler.linear_warmup_schedule(-1, 10, 0.04, 0.07)
    assert scheduler.cosine_schedule(0, 100, 0.992, 1.0) == pytest.approx(0.992)
    assert scheduler.cosine_schedule(100, 100, 0.992, 1.0) == 1.0
    assert scheduler.cosine_schedule(99, 100, 0.992, 1.0) == pytest.approx(1.0)
    for s in (0, 1, 7, 50, 99):
        assert scheduler.cosine_schedule(s, 100, 0.04, 0.4) == pytest.approx(O.cosine_schedule(s, 100, 0.04, 0.4))
    # reference test (tests/_methods/dinov2/test_dinov2.py:137-224): warmup 2 -> lr/2 after the first step
    assert scheduler.cosine_warmup_factor(0, 2, 10, 0.01) == pytest.approx(0.5)
    assert scheduler.cosine_warmup_factor(1, 2, 10, 0.01) == pytest.approx(1.0)
    assert scheduler.cosine_warmup_factor(10, 2, 10, 0.01) == pytest.approx(0.01)


@pytest.mark.parametrize("M,w0,off,aa", [(14, 6, 0.1, False), (16, 7, 0.1, False), (14, 6, 0.0, True), (37, 7, 0.1, True)])
def test_pos_embed_operator_matches_interpolate(M, w0, off, aa):
    x = torch.randn(1, 5, M, M)
    kw = dict(scale_factor=((w0 + off) / M, (w0 + off) / M)) if off else dict(size=(w0, w0))
    y = F.interpolate(x, mode="bicubic", antialias=aa, **kw)
    W = torch.from_numpy(pos_embed_operator(M, w0, w0, off, aa))
    y2 = (W @ x.reshape(5, M * M).t()).t().reshape(1, 5, w0, w0)
    torch.testing.assert_close(y2, y, rtol=1e-4, atol=1e-5)


def _tiny_method(separate_ibot: bool = False):
    from lightly_train_b200._methods.dinov2.dinov2 import DINOv2, DINOv2AdamWViTArgs, DINOv2Args
    margs = DINOv2Args(hidden_dim=64, dino_bottleneck_dim=32, output_dim=128, ibot_separate_head=separate_ibot)
    mk = dict(img_size=32, patch_size=16, embed_dim=64, depth=2, num_heads=1, init_values=1e-5, drop_path_rate=0.1)
    return DINOv2(margs, DINOv2AdamWViTArgs(), mk, global_batch_size=8, max_steps=10, device="cpu")


@pytest.mark.parametrize("separate_ibot", [False, True])
def test_gradient_arena_splits_into_backbone_and_head_parts(separate_ibot):
    """The data-parallel all-reduce goes out in two parts (heads early, backbone after the backward): the split offset
    must separate exactly the backbone parameters from the head parameters, on a chunk boundary."""
    from lightly_train_b200._arena import CHUNK
    m = _tiny_method(separate_ibot)
    off = m._head_off
    assert 0 < off < m.s_arena.total and off % CHUNK == 0
    for name, (o, n) in m.s_arena.offsets.items():
        assert (o >= off) == name.startswith(("dino_head.", "ibot_head.")), name
        assert o + n <= off or o >= off  # no parameter straddles the split


def test_product_path_fails_loudly_without_a_gpu():
    """No CPU / oracle fallback behind the public step: without CUDA the call raises instead of computing."""
    m = _tiny_method()
    views = [torch.randn(2, 3, 32, 32) for _ in range(2)]
    with pytest.raises((RuntimeError, AssertionError)):
        m.train_step({"views": views})


def test_state_dict_names_and_shapes_match_the_reference_modules(golden_dir):
    """Drop-in boundary (SURVEY 8b / appendix A): the mirror classes expose exactly the reference's parameter names and
    shapes (lists dumped from the imported reference modules by tools/make_golden.py), so its checkpoints load unchanged."""
    import json
    from lightly_train_b200._methods.dinov2.dinov2_head import DINOv2ProjectionHead
    from lightly_train_b200._models.dinov2_vit import DinoVisionTransformer
    ref = json.loads((golden_dir / "ref_state_dict_shapes.json").read_text())
    mine = {
        "vit_small_p16": DinoVisionTransformer(img_size=224, patch_size=16, embed_dim=384, depth=12, num_heads=6,
                                               init_values=1e-5, device="cpu"),
        "vit_base_p14_reg4_swiglu": DinoVisionTransformer(img_size=518, patch_size=14, embed_dim=768, depth=12, num_heads=12,
                                                          init_values=1e-5, num_register_tokens=4, ffn_layer="swiglufused",
                                                          interpolate_antialias=True, interpolate_offset=0.0, device="cpu"),
        "head_384_65536": DINOv2ProjectionHead(384, 65536, hidden_dim=2048, bottleneck_dim=256, device="cpu"),
    }
    for name, mod in mine.items():
        got = {k: list(v.shape) for k, v in mod.state_dict().items()}
        assert got == ref[name], (name, set(got) ^ set(ref[name]))


def test_chunked_block_checkpoint_names_load(golden_dir):
    """Zoo configs with block_chunks > 0 (ViT-L / ViT-g) name their blocks `blocks.{chunk}.{i}.*`; the mirror loads them.
    The checkpoint has the layout of the reference's own DinoVisionTransformer(block_chunks=2) (names and shapes stored by
    tools/make_method_golden.py) and seeded random values."""
    import json

    from lightly_train_b200._models.dinov2_vit import DinoVisionTransformer

    layout = json.loads((golden_dir / "method_boundary.json").read_text())["chunked_vit_state_dict"]
    g = torch.Generator().manual_seed(3)
    r = {k: torch.randn(shape, generator=g) for k, shape in layout}
    assert "blocks.1.3.attn.qkv.weight" in r
    m = DinoVisionTransformer(embed_dim=128, depth=4, num_heads=2, init_values=1e-5, device="cpu")
    res = m.load_state_dict(r, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert torch.equal(m.state_dict()["blocks.3.attn.qkv.weight"], r["blocks.1.3.attn.qkv.weight"])
    assert not m.arena.bf16_valid
