"""-m gpu: the distillation path (BASELINE cfg4; SURVEY 8a rows a16 / a17) -- RoPE kernel, fused KL kernels, the DINOv3
teacher forward on the B200 kernels against the oracle and the reference-generated fixtures, and the whole DistillationV3
step against the reference's OWN method class (stored from a run through oracle/ref_full.py) on identical weights,
inputs and mixup draws."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs CUDA", allow_module_level=True)

from lightly_train_b200 import ops  # noqa: E402
from lightly_train_b200._methods.distillationv3.distillationv3 import DistillationV3, DistillationV3Args  # noqa: E402
from lightly_train_b200._methods.distillationv3.distillationv3_loss import DistillationV3Loss  # noqa: E402
from lightly_train_b200._models.dinov3_vit import DinoV3VisionTransformer, DINOv3ViTModelWrapper  # noqa: E402
from lightly_train_b200._models.torchvision_resnet import EmbeddingModel, ResNetModelWrapper  # noqa: E402
from oracle import dinov3_oracle as D3  # noqa: E402
from oracle import distillationv3_oracle as DO  # noqa: E402
from tests.golden import recipes as R  # noqa: E402

dev = "cuda"


def test_rope_kernel_matches_reference_formula():
    B, N, prefix, h = 3, 1 + 4 + 35, 5, 2
    g = torch.Generator().manual_seed(1)
    qkv = torch.randn(B * N, 3 * h * 64, generator=g).to(dev, torch.bfloat16)
    cfg = D3.Dinov3Config(embed_dim=128, num_heads=2)
    sin, cos = D3.rope_sincos(cfg, 5, 7)
    want = qkv.clone().float().view(B, N, 3, h, 64)
    for which in (0, 1):
        x = want[:, prefix:, which]                                   # [B, P, h, 64]
        want[:, prefix:, which] = D3._rope_apply(x, sin[None, :, None].to(dev), cos[None, :, None].to(dev))
    got = qkv.clone()
    ops.rope_apply(got, B, N, prefix, h, sin.to(dev).contiguous(), cos.to(dev).contiguous())
    want_bf = want.view(B * N, -1).bfloat16()
    assert torch.equal(got.view(B, N, 3, h, 64)[:, :prefix], qkv.view(B, N, 3, h, 64)[:, :prefix])   # cls / storage untouched
    assert torch.equal(got.view(B, N, 3, h, 64)[:, :, 2], qkv.view(B, N, 3, h, 64)[:, :, 2])          # v untouched
    assert (got.float() - want_bf.float()).abs().max().item() <= 2e-2  # one bf16 ulp at |x| ~ 3 (fma vs mul+add)
    assert (got.float() - want_bf.float()).abs().mean().item() < 2e-4


def test_kl_loss_kernels_match_oracle_and_reference_fixture(golden_dir):
    ref = torch.load(golden_dir / "distill_v3_loss.pt")
    tg, tl, sg, sl, q = (t.to(dev) for t in R.distill_case_inputs())
    sg.requires_grad_(True); sl.requires_grad_(True)
    lg, ll = DistillationV3Loss(0.07, 0.05)(tg, tl, sg, sl, q)
    (lg + 2 * ll).backward()
    og, ol = DO.distillation_v3_loss(tg.cpu(), tl.cpu(), sg.detach().cpu(), sl.detach().cpu(), q.cpu(), 0.07, 0.05)
    assert abs(float(lg) - float(og)) < 1e-5 and abs(float(ll) - float(ol)) < 1e-5
    assert abs(float(lg) - float(ref["loss_global"])) < 1e-5 and abs(float(ll) - float(ref["loss_local"])) < 1e-5
    torch.testing.assert_close(sg.grad.cpu(), ref["d_student_global"], rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(sl.grad.cpu(), ref["d_student_local"], rtol=1e-4, atol=1e-6)
    # the queue-sized row path (one CTA per row, K > 1024)
    g = torch.Generator().manual_seed(3)
    s, t = torch.randn(37, 8192, generator=g).to(dev), torch.randn(37, 8192, generator=g).to(dev)
    rows, ds = torch.empty(37, device=dev), torch.empty(37, 8192, device=dev)
    ops.kl_rows(s, t, 1 / 0.07, rows, ds)
    sr = s.clone().requires_grad_(True)
    want = (F.softmax(t / 0.07, -1) * (F.log_softmax(t / 0.07, -1) - F.log_softmax(sr / 0.07, -1))).sum(-1)
    want.sum().backward()
    torch.testing.assert_close(rows, want.detach(), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(ds, sr.grad, rtol=1e-3, atol=1e-5)


def test_dinov3_teacher_forward_parity(golden_dir):
    """RoPE on a NON-SQUARE patch grid (14 x 6), storage tokens, masked k bias, eps 1e-5, 30 % masked tokens."""
    ref = torch.load(golden_dir / "dinov3_tiny.pt")
    cfg = R.dinov3_tiny_cfg()
    sd = R.det_dinov3_state(cfg, seed=14)
    vit = DinoV3VisionTransformer(img_size=224, patch_size=cfg.patch_size, embed_dim=cfg.embed_dim, depth=cfg.depth,
                                  num_heads=cfg.num_heads, ffn_ratio=cfg.ffn_ratio, layerscale_init=cfg.layerscale_init,
                                  norm_layer="layernormbf16", n_storage_tokens=cfg.n_storage_tokens, mask_k_bias=True,
                                  pos_embed_rope_base=cfg.rope_base, pos_embed_rope_dtype="fp32")
    r = vit.load_state_dict(sd, strict=False)
    assert not r.unexpected_keys and all(k.endswith("bias_mask") or k == "rope_embed.periods" for k in r.missing_keys), r
    x, masks = R.dinov3_case_inputs()
    o = vit.forward_features(x.to(dev), masks.to(dev))
    want = D3.forward_features(sd, cfg, x, masks)
    for mine, key in (("x_norm_clstoken", "cls"), ("x_storage_tokens", "storage"), ("x_norm_patchtokens", "patch")):
        got = o[mine].float().cpu()
        assert (got - want[key]).abs().max().item() < 8e-2, key     # bf16 GEMMs vs the fp32 oracle, O(1)..O(3) features
        assert (got - want[key]).abs().mean().item() < 6e-3, key
        assert (got - ref[key]).abs().mean().item() < 6e-3, key     # the reference module's own output
    # checkpoint names: the reference state_dict (incl. its buffers) loads strictly
    names = set(vit.state_dict().keys())
    assert {"rope_embed.periods", "blocks.0.attn.qkv.bias_mask", "storage_tokens", "cls_token", "mask_token"} <= names


def test_distillation_step_matches_reference_method(golden_dir):
    """Two training_step_impl calls and the backward of the second against the reference's own DistillationV3 (stored by
    tools/make_method_golden.py): same teacher and projection-head weights (recipes), same ResNet-18 initialisation
    (torch.manual_seed(0)), same input and mixup seeds.  Gradients are compared at the stored elements."""
    import torchvision

    ref = torch.load(golden_dir / "distillation_v3_step.pt")
    tvit = DinoV3VisionTransformer(**R.DISTILL_TEACHER_KW)
    r = tvit.load_state_dict(R.det_dinov3_state(R.dinov3_tiny_cfg(), seed=15), strict=False)
    assert not r.unexpected_keys and all(k.endswith("bias_mask") or k == "rope_embed.periods" for k in r.missing_keys), r
    torch.manual_seed(0)
    resnet = torchvision.models.resnet18()
    student = EmbeddingModel(ResNetModelWrapper(resnet)).to(dev)
    mm = DistillationV3(DistillationV3Args(queue_size=64), None, student, 4, 3, teacher_embedding_model=DINOv3ViTModelWrapper(tvit)).to(dev)
    for n in ("student_projection_head_global", "student_projection_head_local"):
        R.det_fill_(getattr(mm, n), seed=16)
    x = R.distill_step_input()
    for step in range(2):  # second step: the queue already holds the first batch
        torch.manual_seed(100 + step)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            mres = mm.training_step_impl({"views": [x.to(dev)]}, 0)
        want = ref["steps"][step]
        for k in ("global_loss", "local_loss"):
            a, b = float(mres.log_dict["train_loss/" + k]), want[k]
            assert abs(a - b) < 2e-2 * max(1.0, abs(b)), (step, k, a, b)  # bf16 autocast student + bf16 teacher vs fp32 reference
        q = torch.zeros_like(mm.teacher_queue, device="cpu")
        q[:want["queue_head"].shape[0]] = want["queue_head"]  # the rest of the reference queue is still zero
        assert (mm.teacher_queue.cpu() - q).abs().max().item() < 3e-2
    mres.loss.backward()
    res = mm.student_embedding_model.wrapped_model.get_model()
    got = {"head_global": mm.student_projection_head_global.weight.grad, "layer4.1.conv2": res.layer4[1].conv2.weight.grad,
           "conv1": res.conv1.weight.grad}
    got = {k: v.float().cpu().flatten()[R.sample_index(v.numel(), ref["grads"][k]["sample"].numel())] for k, v in got.items()}
    gb = ref["grads"]["head_global"]["sample"]
    assert ((got["head_global"] - gb).norm() / gb.norm()).item() < 0.1
    # deep in the student (bf16 autocast convs + BatchNorm over 4 images vs the fp32 reference): direction, not digits
    cos = torch.nn.functional.cosine_similarity
    assert cos(got["layer4.1.conv2"], ref["grads"]["layer4.1.conv2"]["sample"], dim=0).item() > 0.9
    assert cos(got["conv1"], ref["grads"]["conv1"]["sample"], dim=0).item() > 0.6


def test_sibling_distillation_losses():
    """Distillation v1 (queue KL, LT/_methods/distillation/distillation_loss.py) and v2 (MSE, distillationv2_loss.py) on the
    fused kernels against the torch statement of the reference modules' forward, values and student gradients."""
    from lightly_train_b200._methods.distillation.distillation_loss import DistillationLoss
    from lightly_train_b200._methods.distillationv2.distillationv2_loss import DistillationV2Loss
    tg, tl, sg, sl, q = (t.to(dev) for t in R.distill_case_inputs())
    s1 = sg.clone().requires_grad_(True)
    l1 = DistillationLoss(0.07)(tg, s1, q)
    l1.backward()
    s2 = sg.clone().requires_grad_(True)
    want = F.kl_div(F.log_softmax(s2 @ q.t() / 0.07, -1), F.softmax(tg @ q.t() / 0.07, -1), reduction="batchmean")
    want.backward()
    assert abs(float(l1) - float(want)) < 1e-5
    torch.testing.assert_close(s1.grad, s2.grad, rtol=1e-4, atol=1e-6)
    a = sl.clone().requires_grad_(True)
    l2 = DistillationV2Loss()(tl, a)
    l2.backward()
    b = sl.clone().requires_grad_(True)
    w2 = F.mse_loss(tl, b)
    w2.backward()
    assert abs(float(l2) - float(w2)) < 1e-6
    torch.testing.assert_close(a.grad, b.grad, rtol=1e-5, atol=1e-8)
