"""Generate tests/golden/* by running the REFERENCE's own modules (imported in place from a lightly-train source tree
via oracle/ref_shim.py) on seeded inputs.  The fixtures it writes are committed and are what the oracle (and through it
the CUDA path) is pinned against; the tests themselves never need the reference.

    LIGHTLY_TRAIN_SRC=<lightly-train checkout>/src python tools/make_golden.py

Glue that cannot be imported (the LightningModule shell, LT/_methods/dinov2/dinov2.py:259-519, needs
pytorch_lightning/lightly) is composed here from the reference's modules in the same order; KoLeoLoss
(third-party `lightly`) is absent, so koleo values in the fixtures come from the restated definition and are
marked "unpinned".
"""
from __future__ import annotations

import json
import random
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from oracle import ref_shim  # noqa: E402
from oracle import dinov2_oracle as O  # noqa: E402  (only koleo_loss + det_* helpers are used from here)
from tests.golden import recipes as R  # noqa: E402

OUT = ROOT / "tests" / "golden"


def ref_kats(m) -> dict:
    """Re-run the reference's own known-answer tests with the reference's own classes."""
    out = {}
    dl = m.loss.DINOLoss(out_dim=2, student_temp=0.1, center_momentum=0.9)
    t = torch.tensor([[0.1, 0.2], [0.3, 0.4], [0.5, 0.6]])
    s = [torch.tensor([[0.7, 0.8], [0.9, 1.0], [1.1, 1.2]]) for _ in range(2)]
    tp = dl.softmax_center_teacher(t, teacher_temp=0.04)
    dl.update_center(t)
    out["dino_forward"] = float(dl.forward(s, [tp, tp]))  # reference asserts approx 1.5565
    dl.apply_center_update()
    out["dino_center_after"] = dl.center.flatten().tolist()

    il = m.loss.IBOTPatchLoss(patch_out_dim=2, student_temp=0.2, center_momentum=0.9)
    mask = torch.tensor([[True, False, True, False], [False, False, False, True], [False, False, False, False]])
    tp = il.softmax_center_teacher(t.unsqueeze(0), teacher_temp=0.1)
    il.update_center(t.unsqueeze(0))
    out["ibot_forward_masked"] = float(il.forward_masked(
        teacher_patch_tokens_masked=tp, student_patch_tokens_masked=s[0], student_masks_flat=mask))  # 0.4057

    dl2 = m.loss.DINOLoss(out_dim=2)
    dl2.update_center(torch.ones(4, 2) * 2)
    dl2.apply_center_update()
    out["center_momentum"] = dl2.center.flatten().tolist()  # 0.2

    a = torch.nn.Linear(2, 2, bias=False)
    b = torch.nn.Linear(2, 2, bias=False)
    with torch.no_grad():
        a.weight.copy_(torch.tensor([[3.0, 4.0], [5.0, 6.0]]))
        b.weight.copy_(torch.tensor([[1.0, 2.0], [3.0, 4.0]]))
    m.torch_helpers.update_momentum(model=a, model_ema=b, m=0.25)
    out["ema"] = b.weight.tolist()  # [[2.5,3.5],[4.5,5.5]]

    out["linear_warmup"] = [m.scheduler.linear_warmup_schedule(s_, 37500, 0.04, 0.07) for s_ in (0, 100, 37500, 50000)]
    return out


def build_ref_vit(m, cfg: O.ViTConfig, sd):
    vit = m.vit.DinoVisionTransformer(
        img_size=cfg.img_size, patch_size=cfg.patch_size, embed_dim=cfg.embed_dim, depth=cfg.depth,
        num_heads=cfg.num_heads, mlp_ratio=cfg.mlp_ratio, init_values=cfg.init_values, block_chunks=0,
        num_register_tokens=cfg.num_register_tokens, interpolate_offset=cfg.interpolate_offset,
        interpolate_antialias=cfg.interpolate_antialias, ffn_layer=cfg.ffn_layer,
        block_fn=__import__("functools").partial(m.vit.Block, attn_class=m.vit.MemEffAttention))
    missing = vit.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return vit


def build_ref_head(m, cfg: O.HeadConfig, sd):
    h = m.head.DINOv2ProjectionHead(in_dim=cfg.in_dim, out_dim=cfg.out_dim, hidden_dim=cfg.hidden_dim,
                                    bottleneck_dim=cfg.bottleneck_dim)
    h.load_state_dict(sd, strict=True)
    return h


def vit_case(m) -> dict:
    cfg = R.VIT_TINY
    sd = R.det_vit_state(cfg, seed=11)
    vit = build_ref_vit(m, cfg, sd).eval()
    xg, xl, masks = R.vit_case_inputs()
    with torch.no_grad():
        g = vit(xg, masks, is_training=True)
        g_nomask = vit(xg, None, is_training=True)
        l = vit(xl, None, is_training=True)
    return {
        "g_cls": g["x_norm_clstoken"], "g_patch": g["x_norm_patchtokens"], "g_prenorm": g["x_prenorm"],
        "g_nomask_cls": g_nomask["x_norm_clstoken"],
        "l_cls": l["x_norm_clstoken"], "l_patch": l["x_norm_patchtokens"],
        "pos_embed_96": vit.interpolate_pos_encoding(torch.zeros(1, 37, cfg.embed_dim), 96, 96),
    }


def vit_reg_case(m) -> dict:
    """register tokens + antialiased interpolation + no interpolate offset variant (cfg3-style options)."""
    cfg = R.VIT_TINY_REG
    sd = R.det_vit_state(cfg, seed=12)
    vit = build_ref_vit(m, cfg, sd).eval()
    xg, xl, masks = R.vit_case_inputs()
    with torch.no_grad():
        l = vit(xl, None, is_training=True)
        g = vit(xg, masks, is_training=True)
    return {"l_cls": l["x_norm_clstoken"], "g_cls": g["x_norm_clstoken"], "g_patch": g["x_norm_patchtokens"]}


def vit_swiglu_case(m) -> dict:
    """SwiGLU FFN (w12 / w3, hidden = round8(2/3 * 4D)) + register tokens: forward features and every parameter gradient."""
    cfg = R.VIT_TINY_SWIGLU
    sd = R.det_vit_state(cfg, seed=13)
    vit = build_ref_vit(m, cfg, sd).train()  # drop_path_rate = 0: train() only enables the masks path
    xg, xl, masks = R.vit_case_inputs()
    g = vit(xg, masks, is_training=True)
    cot = R.vit_swiglu_cotangents()
    ((g["x_norm_patchtokens"] * cot[0]).sum() + (g["x_norm_clstoken"] * cot[1]).sum()).backward()
    out = {"g_cls": g["x_norm_clstoken"].detach(), "g_patch": g["x_norm_patchtokens"].detach()}
    out.update({"grad." + k: p.grad.clone() for k, p in vit.named_parameters() if p.grad is not None})
    return out


def state_dict_shapes(m) -> dict:
    """Parameter names and shapes of the reference modules (drop-in boundary, SURVEY appendix A)."""
    import functools

    def vit(**kw):
        v = m.vit.DinoVisionTransformer(block_chunks=0, block_fn=functools.partial(m.vit.Block, attn_class=m.vit.MemEffAttention), **kw)
        return {k: list(t.shape) for k, t in v.state_dict().items()}

    h = m.head.DINOv2ProjectionHead(in_dim=384, out_dim=65536, hidden_dim=2048, bottleneck_dim=256)
    return {
        "vit_small_p16": vit(img_size=224, patch_size=16, embed_dim=384, depth=12, num_heads=6, init_values=1e-5),
        "vit_base_p14_reg4_swiglu": vit(img_size=518, patch_size=14, embed_dim=768, depth=12, num_heads=12, init_values=1e-5,
                                        num_register_tokens=4, ffn_layer="swiglufused", interpolate_antialias=True,
                                        interpolate_offset=0.0),
        "head_384_65536": {k: list(t.shape) for k, t in h.state_dict().items()},
    }


def distill_v3_case() -> dict:
    """DistillationV3Loss (temperatures 0.07 / 0.05): both KL terms and the gradients wrt the student features."""
    from lightly_train._methods.distillationv3.distillationv3_loss import DistillationV3Loss  # type: ignore
    tg, tl, sg, sl, q = R.distill_case_inputs()
    sg.requires_grad_(True); sl.requires_grad_(True)
    lg, ll = DistillationV3Loss(0.07, 0.05)(tg, tl, sg, sl, q)
    (lg + 2 * ll).backward()
    return {"loss_global": lg.detach(), "loss_local": ll.detach(), "d_student_global": sg.grad.clone(),
            "d_student_local": sl.grad.clone()}


def dinov3_case() -> dict:
    """DINOv3 ViT (RoPE on patch tokens, 4 storage tokens, masked k bias, LayerNorm eps 1e-5) in eval mode = the teacher
    forward of the distillation method: features of a non-square masked input."""
    from lightly_train._models.dinov3.dinov3_src.models import vision_transformer as v3  # type: ignore
    cfg = R.dinov3_tiny_cfg()
    vit = v3.DinoVisionTransformer(img_size=224, patch_size=cfg.patch_size, embed_dim=cfg.embed_dim, depth=cfg.depth,
                                   num_heads=cfg.num_heads, ffn_ratio=cfg.ffn_ratio, layerscale_init=cfg.layerscale_init,
                                   norm_layer="layernormbf16", n_storage_tokens=cfg.n_storage_tokens, mask_k_bias=True,
                                   pos_embed_rope_base=cfg.rope_base, pos_embed_rope_normalize_coords="separate",
                                   pos_embed_rope_dtype="fp32", pos_embed_rope_rescale_coords=2.0)
    vit.init_weights()  # fills rope periods and the k-bias mask
    sd = R.det_dinov3_state(cfg, seed=14)
    r = vit.load_state_dict(sd, strict=False)
    assert not r.unexpected_keys and all(k.endswith("bias_mask") or k == "rope_embed.periods" for k in r.missing_keys), r
    vit.eval()
    x, masks = R.dinov3_case_inputs()
    with torch.no_grad():
        o = vit.forward_features(x, masks)
    return {"cls": o["x_norm_clstoken"], "storage": o["x_storage_tokens"], "patch": o["x_norm_patchtokens"],
            "prenorm": o["x_prenorm"]}


def vit_autocast_case(m) -> dict:
    """The reference ViTs under REAL bf16 autocast (torch.autocast("cpu", bfloat16): the same op policy family as the CUDA
    autocast the training runs under) -- pins the oracle's autocast=True emulation, which the GPU parity bars rely on."""
    out = {}
    xg, _, masks = R.vit_case_inputs()
    for name, cfg, seed in (("mlp", R.VIT_TINY, 11), ("swiglu", R.VIT_TINY_SWIGLU, 13)):
        vit = build_ref_vit(m, cfg, R.det_vit_state(cfg, seed=seed)).eval()
        with torch.no_grad(), torch.autocast("cpu", dtype=torch.bfloat16):
            g = vit(xg, masks, is_training=True)
        out[name + "_cls"] = g["x_norm_clstoken"].float()
        out[name + "_patch0"] = g["x_norm_patchtokens"][0].float()
    return out


def head_case(m) -> dict:
    cfg = R.HEAD_TINY
    sd = R.det_head_state(cfg, seed=21)
    h = build_ref_head(m, cfg, sd)
    x = R.head_case_input()
    x.requires_grad_(True)
    y = h(x)
    (y * R.head_case_cotangent()).sum().backward()
    grads = {k: p.grad.clone() for k, p in h.named_parameters()}
    return {"logits": y.detach(), "dx": x.grad.clone(), **{"grad." + k: v for k, v in grads.items()}}


def masks_case(m) -> dict:
    out = {}
    for seed, (n_crops, hw) in enumerate([(8, 14), (128, 14), (6, 16)]):
        random.seed(1234 + seed)
        gen = m.utils.MaskingGenerator(input_size=(hw, hw), max_num_patches=int(0.5 * hw * hw))
        res = m.utils.create_collated_masks(mask_ratio_min=0.1, mask_ratio_max=0.5,
                                            n_masked_crops=int(n_crops * 0.5), n_crops=n_crops, mask_generator=gen)
        out[f"case{seed}"] = {"seed": 1234 + seed, "n_crops": n_crops, "hw": hw,
                              "collated_masks": res["collated_masks"], "mask_indices_list": res["mask_indices_list"],
                              "masks_weight": res["masks_weight"]}
    return out


def loss_case(m) -> dict:
    """Loss functions on random logits, both centering methods, K small."""
    g = torch.Generator().manual_seed(31)
    K, B, Mrows = 512, 6, 11
    t_cls = torch.randn(2 * B, K, generator=g)
    t_patch = torch.randn(Mrows, K, generator=g)
    s_g = torch.randn(2 * B, K, generator=g)
    s_l = torch.randn(4 * B, K, generator=g)
    s_patch = torch.randn(Mrows, K, generator=g)
    w = torch.rand(Mrows, generator=g)
    dl = m.loss.DINOLoss(out_dim=K)
    il = m.loss.IBOTPatchLoss(patch_out_dim=K)
    dl.center.copy_(torch.randn(1, K, generator=g) * 0.1)
    il.center.copy_(torch.randn(1, 1, K, generator=g) * 0.1)
    out = {"t_cls": t_cls, "t_patch": t_patch, "s_g": s_g, "s_l": s_l, "s_patch": s_patch, "w": w,
           "center_dino": dl.center.clone(), "center_ibot": il.center.clone()}
    p_cls = dl.softmax_center_teacher(t_cls, 0.05)
    p_patch = il.softmax_center_teacher(t_patch.unsqueeze(0), 0.05).squeeze(0)
    dl.update_center(t_cls)
    il.update_center(t_patch.unsqueeze(0))
    out["p_cls"], out["p_patch"] = p_cls, p_patch
    out["loss_global"] = dl.forward([s_g], [p_cls])
    out["loss_local"] = dl.forward(s_l.chunk(4), list(p_cls.view(2, B, K)))
    masks_flat = torch.zeros(2 * B, 7, dtype=torch.bool)
    out["loss_ibot"] = il.forward_masked(s_patch, p_patch, student_masks_flat=masks_flat, n_masked_patches=Mrows,
                                         masks_weight=w)
    dl.apply_center_update()
    il.apply_center_update()
    out["center_dino_after"], out["center_ibot_after"] = dl.center.clone(), il.center.clone()
    out["sk_cls"] = dl.sinkhorn_knopp_teacher(t_cls, 0.05)
    out["sk_patch"] = il.sinkhorn_knopp_teacher(t_patch, 0.05, n_masked_patches_tensor=torch.tensor([Mrows]))
    return out


def step_autocast_case(m) -> dict:
    """Loss terms and logits of the softmax / shared-head step with the reference modules under real bf16 autocast (CPU)."""
    full = step_case(m, "softmax", False, autocast=True)
    keep = ("loss", "dino_global_loss", "dino_local_loss", "ibot_loss", "koleo_loss", "t_cls_logits", "s_cls_logits_g")
    return {k: full[k].float() for k in keep}


def step_case(m, center_method: str, separate: bool, autocast: bool = False) -> dict:
    """Full loss evaluation + backward with the reference modules, glue per dinov2.py:259-519."""
    cfg = R.step_config(center_method, separate)
    st = R.det_step_state(cfg, seed=41)
    views, masks, idx, w = R.step_case_inputs(cfg)
    teacher_temp = 0.05

    def mk(prefix_sd):
        vit = build_ref_vit(m, cfg.vit, O._sub(prefix_sd, "backbone."))
        dino = build_ref_head(m, cfg.head, O._sub(prefix_sd, "dino_head."))
        ibot = build_ref_head(m, cfg.head, O._sub(prefix_sd, "ibot_head.")) if separate else dino
        return vit, dino, ibot

    s_vit, s_dino, s_ibot = mk(st["student"])
    t_vit, t_dino, t_ibot = mk(st["teacher"])
    t_vit.eval(); t_dino.eval(); t_ibot.eval()
    s_vit.train(); s_dino.train(); s_ibot.train()  # drop_path_rate = 0 -> plain residual
    K = cfg.head.out_dim
    dl = m.loss.DINOLoss(out_dim=K, student_temp=cfg.student_temp, center_momentum=cfg.center_momentum)
    il = m.loss.IBOTPatchLoss(patch_out_dim=K, student_temp=cfg.student_temp, center_momentum=cfg.center_momentum)
    dl.center.copy_(st["centers"]["dino"]); il.center.copy_(st["centers"]["ibot"])

    B = views[0].shape[0]
    D = cfg.vit.embed_dim
    gv = torch.cat(views[:2])
    n_local = len(views) - 2
    g_terms, l_terms = 2, max(n_local * 2, 1)
    ac = torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast)
    ac.__enter__()  # the fit loop wraps training_step in the precision plugin's autocast context
    with torch.no_grad():
        tt = t_vit(gv, None, is_training=True)
        cls = tt["x_norm_clstoken"]
        cls = torch.cat((cls[B:], cls[:B]))
        cls_after = t_dino(cls)
        patch = tt["x_norm_patchtokens"].flatten(0, 1).index_select(0, idx)
        patch_after = t_ibot(patch)
        if center_method == "softmax":
            cls_c = dl.softmax_center_teacher(cls_after, teacher_temp=teacher_temp).view(2, -1, K)
            dl.update_center(cls_after)
            patch_c = il.softmax_center_teacher(patch_after.unsqueeze(0), teacher_temp=teacher_temp).squeeze(0)
            il.update_center(patch_after.unsqueeze(0))
        else:
            cls_c = dl.sinkhorn_knopp_teacher(cls_after, teacher_temp=teacher_temp).view(2, -1, K)
            patch_c = il.sinkhorn_knopp_teacher(patch_after, teacher_temp=teacher_temp,
                                                n_masked_patches_tensor=torch.tensor([idx.shape[0]]))
    sg = s_vit(gv, masks, is_training=True)
    s_cls = sg["x_norm_clstoken"]
    s_cls_after = s_dino(s_cls)
    s_patch_after = s_ibot(sg["x_norm_patchtokens"].flatten(0, 1).index_select(0, idx))
    dino_global = dl.forward([s_cls_after], [cls_c.flatten(0, 1)]) * 2 / (g_terms + l_terms)
    dino_local = torch.zeros_like(dino_global)
    if n_local:
        sl = s_vit(torch.cat(views[2:]), None, is_training=True)
        s_local_after = s_dino(sl["x_norm_clstoken"])
        dino_local = dl.forward(s_local_after.chunk(n_local), cls_c) / (g_terms + l_terms)
    ibot = il.forward_masked(s_patch_after, patch_c, student_masks_flat=masks, n_masked_patches=idx.shape[0],
                             masks_weight=w)
    koleo = sum(O.koleo_loss(c) for c in s_cls.chunk(2))  # lightly.KoLeoLoss restated (unpinned)
    loss = dino_global + dino_local + ibot + 0.1 * koleo
    ac.__exit__(None, None, None)
    loss.backward()
    out = {"loss": loss.detach(), "dino_global_loss": dino_global.detach(), "dino_local_loss": dino_local.detach(),
           "ibot_loss": ibot.detach(), "koleo_loss": koleo.detach(),
           "t_cls_logits": cls_after, "t_patch_logits": patch_after, "s_cls_logits_g": s_cls_after.detach(),
           "s_patch_logits": s_patch_after.detach()}
    if center_method == "softmax":
        dl.apply_center_update(); il.apply_center_update()
        out["center_dino_after"], out["center_ibot_after"] = dl.center.clone(), il.center.clone()
    mods = {"backbone.": s_vit, "dino_head.": s_dino}
    if separate:
        mods["ibot_head."] = s_ibot
    for pre, mod in mods.items():
        for k, p in mod.named_parameters():
            out["grad." + pre + k] = p.grad.clone() if p.grad is not None else torch.zeros_like(p)
    return out


def main() -> None:
    torch.manual_seed(0)
    torch.set_num_threads(8)
    m = ref_shim.modules()
    OUT.mkdir(parents=True, exist_ok=True)
    (OUT / "ref_kats.json").write_text(json.dumps(ref_kats(m), indent=1))
    torch.save(vit_case(m), OUT / "vit_tiny.pt")
    torch.save(vit_reg_case(m), OUT / "vit_tiny_reg.pt")
    (OUT / "ref_state_dict_shapes.json").write_text(json.dumps(state_dict_shapes(m), indent=0))
    torch.save(vit_swiglu_case(m), OUT / "vit_tiny_swiglu.pt")
    torch.save(vit_autocast_case(m), OUT / "vit_tiny_autocast_cpu.pt")
    torch.save(step_autocast_case(m), OUT / "step_softmax_shared_autocast_cpu.pt")
    torch.save(distill_v3_case(), OUT / "distill_v3_loss.pt")
    torch.save(dinov3_case(), OUT / "dinov3_tiny.pt")
    torch.save(head_case(m), OUT / "head_tiny.pt")
    torch.save(masks_case(m), OUT / "masks.pt")
    torch.save(loss_case(m), OUT / "loss_case.pt")
    for cm, sep in (("softmax", False), ("sinkhorn_knopp", True)):
        torch.save(step_case(m, cm, sep), OUT / f"step_{cm}_{'sep' if sep else 'shared'}.pt")
    for f in sorted(OUT.glob("*")):
        print(f.name, f.stat().st_size)


if __name__ == "__main__":
    main()
