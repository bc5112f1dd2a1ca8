"""-m gpu: the mirror driven the way Lightning drives the reference Method (LT/_methods/method.py:131-148,
LT/_methods/dinov2/dinov2.py:550-660): a plain python loop standing in for the trainer calls the reference's hook names
in automatic-optimisation order.  Also: checkpoint round trip into the reference's own modules, update_momentum with the
reference signature, and the stochastic-depth code paths that draw their own random numbers."""
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs CUDA", allow_module_level=True)

from lightly_train_b200._methods.dinov2.dinov2 import DINOv2, DINOv2AdamWViTArgs, DINOv2Args  # noqa: E402
from lightly_train_b200._models.dinov2_vit import DinoVisionTransformer  # noqa: E402
from lightly_train_b200._torch_helpers import update_momentum  # noqa: E402
from oracle import dinov2_oracle as O  # noqa: E402
from tests import ref_cases as RC  # noqa: E402
from tests.golden import recipes as R  # noqa: E402

dev = "cuda"


def _tiny_method(max_steps=10, **over) -> DINOv2:
    cfg = R.step_config("softmax", False)
    st = R.det_step_state(cfg, seed=41)
    margs = DINOv2Args(hidden_dim=cfg.head.hidden_dim, dino_bottleneck_dim=cfg.head.bottleneck_dim, output_dim=cfg.head.out_dim,
                       warmup_steps=2, student_freeze_last_layer_steps=1, **over)
    mk = dict(img_size=224, patch_size=16, embed_dim=cfg.vit.embed_dim, depth=cfg.vit.depth, num_heads=cfg.vit.num_heads,
              init_values=cfg.vit.init_values, drop_path_rate=0.0)
    m = DINOv2(margs, DINOv2AdamWViTArgs(), mk, global_batch_size=1024, max_steps=max_steps, device=dev)
    m.s_arena.load_from(st["student"]); m.t_arena.load_from(st["teacher"])
    m.dino_loss.center.copy_(st["centers"]["dino"]); m.ibot_loss.center.copy_(st["centers"]["ibot"])
    return m


def _lightning_like_fit(m: DINOv2, batches, steps: int):
    """What pytorch_lightning's fit loop does per batch under automatic optimisation, with the hook names the reference
    method implements; `loss.backward()` goes through the autograd bridge (gradients are already in param.grad)."""
    (opt,), (sch,) = m.configure_optimizers()
    losses = []
    for i in range(steps):
        batch = batches[i % len(batches)]
        opt.zero_grad()
        loss = m.training_step(batch, i)                     # Method.training_step: step + log / log_dict(sync_dist)
        DINOv2.loss_for_autograd(m._last_result).backward()  # trainer-side backward: a no-op on the bridge leaf
        m.on_before_optimizer_step(opt)
        m.configure_gradient_clipping(opt, gradient_clip_val=None, gradient_clip_algorithm=None)
        opt.step()
        sch["scheduler"].step()
        m.trainer.global_step += 1
        m.on_train_batch_end(loss, batch, i)
        losses.append(float(loss))
    return losses


def test_lightning_shaped_loop_equals_train_step():
    cfg = R.step_config("softmax", False)
    views, masks, idx, w = R.step_case_inputs(cfg)
    batch = {"views": [v.to(dev) for v in views], "masks": {"collated_masks": masks, "mask_indices_list": idx, "masks_weight": w}}
    a, b = _tiny_method(), _tiny_method()
    la = _lightning_like_fit(a, [batch], 3)
    lb = [float(b.train_step(batch).loss) for _ in range(3)]
    torch.cuda.synchronize()
    # steps 0 and 1 see identical weights (the warm-up lr of step 0 is 0); step 2 sees the first real Adam update, which is
    # lr * g/|g|: run-to-run reordering of the fp32 split-K atomics flips it for noise-level gradients (observed 7e-4 on the
    # loss between two identical runs), so only steps 0-1 are compared tightly.  The update rule itself is pinned by
    # test_optimizer_ema_step_matches_oracle and the hook order by test_ema_hook_order_and_unfused_update_momentum.
    assert la[:2] == pytest.approx(lb[:2], rel=1e-5)
    assert la[2] == pytest.approx(lb[2], rel=3e-3)
    # fp32 split-K atomics reorder the wgrad sums run to run and Adam's first steps are lr * g/|g|: elements whose gradient
    # sits at rounding-noise level can move by up to ~lr (here 2e-3) differently in two runs; everything else agrees tightly
    d = (a.s_arena.fp32 - b.s_arena.fp32).abs()
    # (a systematic difference -- a wrong lr / weight-decay / momentum index -- moves EVERY element by ~lr: mean ~1e-3)
    assert d.max().item() < 3 * a.base_lr and d.mean().item() < 2e-5 and (d > 1e-5).float().mean().item() < 0.15
    assert (a.t_arena.fp32 - b.t_arena.fp32).abs().max().item() < 1e-4
    assert a.trainer.global_step == b.trainer.global_step == 3
    for k in ("train_loss", "train_loss/dino_global_loss", "train_loss/dino_local_loss", "train_loss/ibot_loss", "train_loss/koleo_loss"):
        assert k in a.logged and torch.isfinite(a.logged[k]).item()
    # hooks visible through the optimizer shim like through a torch optimizer
    (opt,), (sch,) = a.configure_optimizers()
    names = [g["name"] for g in opt.param_groups]
    assert "cls_token" in names and any("last_layer" in n for n in names)
    assert len(sch["scheduler"].get_last_lr()) == len(opt.param_groups)


def test_ema_hook_order_and_unfused_update_momentum():
    """The fused sweep applies the EMA with the momentum of global_step + 1 (Lightning increments before
    on_train_batch_end); running the sweep without its EMA part and then the reference-signature update_momentum in the
    hook must give the same teacher."""
    cfg = R.step_config("softmax", False)
    views, masks, idx, w = R.step_case_inputs(cfg)
    batch = {"views": [v.to(dev) for v in views], "masks": {"collated_masks": masks, "mask_indices_list": idx, "masks_weight": w}}
    a, b = _tiny_method(), _tiny_method()
    t_before = a.t_arena.fp32.clone()
    a.train_step(batch)
    # b: same step, EMA through the hook
    b.training_step_impl(batch, 0)
    (opt,), (sch,) = b.configure_optimizers()
    b.on_before_optimizer_step(opt); b.configure_gradient_clipping(opt)
    b._fused_sweep(opt, b.base_lr * sch["scheduler"].factor(), fuse_ema=False)
    sch["scheduler"].step(); b.trainer.global_step += 1
    assert torch.equal(b.t_arena.fp32, t_before)  # teacher untouched so far
    b.on_train_batch_end(None, batch, 0)
    torch.cuda.synchronize()
    # each run against ITS OWN student (the two students differ by run-to-run atomics noise through Adam's first step, which
    # the EMA passes on scaled by 1 - m): exact identity; across the runs only the noise bound
    m = O.cosine_schedule(1, 10, a.method_args.momentum_start, a.method_args.momentum_end)
    want = t_before * m + a.s_arena.fp32 * (1 - m)
    assert (a.t_arena.fp32 - want).abs().max().item() < 1e-6
    want_b = t_before * m + b.s_arena.fp32 * (1 - m)
    assert (b.t_arena.fp32 - want_b).abs().max().item() < 1e-6
    assert (a.t_arena.fp32 - b.t_arena.fp32).abs().max().item() < 3 * a.base_lr * (1 - m) + 1e-6
    # reference signature on arbitrary arena-backed modules (LT/_torch_helpers.py:89-96)
    t2 = b.t_arena.fp32.clone()
    update_momentum(b.student_head, b.teacher_head, 0.5)
    off = b._head_off
    assert torch.equal(b.t_arena.fp32[:off], t2[:off])
    assert torch.allclose(b.t_arena.fp32[off:], 0.5 * t2[off:] + 0.5 * b.s_arena.fp32[off:], atol=1e-7)
    assert torch.equal(b.t_arena.bf16[off:], b.t_arena.fp32[off:].bfloat16())


def test_checkpoint_resume_is_exact():
    """Optimizer moments, AdamW step count, scheduler epoch and global_step round-trip through the Lightning-layout
    checkpoint: a resumed run continues exactly like the uninterrupted one (same graph-free schedule, same batch)."""
    cfg = R.step_config("softmax", False)
    views, masks, idx, w = R.step_case_inputs(cfg)
    batch = {"views": [v.to(dev) for v in views], "masks": {"collated_masks": masks, "mask_indices_list": idx, "masks_weight": w}}
    a = _tiny_method()
    a.train_step(batch); a.train_step(batch)
    a.dino_loss.apply_center_update(); a.ibot_loss.apply_center_update()
    ck = a.checkpoint()
    assert set(ck) == {"state_dict", "optimizer_states", "lr_schedulers", "global_step"} and ck["global_step"] == 2
    b = _tiny_method()
    b.load_checkpoint(ck)
    assert not b.s_arena.bf16_valid and not b.t_arena.bf16_valid
    assert b._opt_step == 2 and b.trainer.global_step == 2
    assert torch.equal(a.s_arena.exp_avg, b.s_arena.exp_avg) and torch.equal(a.s_arena.fp32, b.s_arena.fp32)
    ra, rb = a.train_step(batch), b.train_step(batch)
    torch.cuda.synchronize()
    assert abs(float(ra.loss) - float(rb.loss)) < 1e-5 * abs(float(ra.loss))
    # identical state going in; the step itself reorders fp32 atomics run to run (see the Lightning-loop test): elements with
    # noise-level gradients may differ by ~lr, everything else agrees tightly
    d = (a.s_arena.fp32 - b.s_arena.fp32).abs()
    assert d.max().item() < 3 * a.base_lr and d.mean().item() < 2e-5 and (d > 1e-5).float().mean().item() < 0.15


def test_checkpoint_round_trip_into_reference_modules(golden_dir):
    """1 optimisation step on CUDA -> state_dict() in exactly the reference DINOv2 method's checkpoint layout (names, order
    and shapes stored from the reference's own class by tools/make_method_golden.py, so its load_state_dict(strict=True)
    takes it) -> the fp32 ViT forward on those weights (the oracle, pinned against the reference modules by
    tests/test_oracle_goldens.py) reproduces the CUDA teacher/student features."""
    import json

    case = RC.TINY
    cfg = RC.oracle_cfg(case)
    st = R.det_step_state(cfg, seed=41)
    mk = {k: v for k, v in case.vit.items() if k != "block_chunks"}
    m = DINOv2(DINOv2Args(**dict(dict(warmup_steps=2, student_freeze_last_layer_steps=1), **case.method)), DINOv2AdamWViTArgs(),
               mk, case.batch, 3, max_steps=100, device=dev)
    RC.load_oracle_state(m, st["student"], st["teacher"], st["centers"])
    views = RC.make_views(case)
    random.seed(3)
    m.train_step({"views": [v.to(dev) for v in views]})
    m.dino_loss.apply_center_update(); m.ibot_loss.apply_center_update()
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    layout = json.loads((golden_dir / "method_boundary.json").read_text())["tiny_method_state_dict"]
    assert [[k, list(v.shape)] for k, v in sd.items()] == layout
    student, teacher, _ = RC.oracle_state(sd, cfg.ibot_separate_head)
    x = views[0]
    with torch.no_grad():
        for side, w in (("teacher", teacher), ("student", student)):
            want = O.vit_forward_features(O._sub(w, "backbone."), cfg.vit, x)["cls"]
            got = getattr(m, f"{side}_embedding_model").wrapped_model.get_model().forward_features(x.to(dev))["x_norm_clstoken"]
            assert (got.float().cpu() - want).abs().max().item() < 5e-2, side  # bf16 GEMMs vs fp32, O(1) features
            assert (got.float().cpu() - want).abs().mean().item() < 5e-3, side
    # the step really moved the student away from the teacher-initialised weights
    assert (sd["student_embedding_model.wrapped_model._model.blocks.0.attn.qkv.weight"]
            - st["student"]["backbone.blocks.0.attn.qkv.weight"]).abs().max().item() > 0


def test_stochastic_depth_rng_paths():
    """The code that draws the stochastic-depth randomness itself (bench path): per-sample DropPath for rates <= 0.1
    (`bern_scales`) and the batch-subset form for rates > 0.1 (layers/block.py:118-141).  Checks the scale statistics and
    that a dropped sample receives NO gradient contribution from the dropped branch."""
    torch.manual_seed(0)
    Bc = 64
    m = DinoVisionTransformer(img_size=32, patch_size=16, embed_dim=128, depth=4, num_heads=2, init_values=1.0,
                              drop_path_rate=0.3, drop_path_uniform=False, requires_grad=True)
    assert [round(r, 3) for r in m.dpr] == [0.0, 0.1, 0.2, 0.3]
    x = torch.randn(Bc, 3, 32, 32, device=dev)
    m.arena.zero_grad()
    ctx = m._fwd(x, None, save=True, drop_path=True)
    blocks = ctx.blocks
    assert blocks[0]["rs1"] is None and blocks[0]["rs2"] is None            # rate 0: no scaling
    # torch.linspace is float32: the second rate is 0.10000000149 > 0.1, so -- exactly like the reference's
    # `sample_drop_ratio > 0.1` test (block.py:104) -- block 1 already takes the batch-subset form
    assert m.dpr[1] > 0.1
    for i, rate in ((1, 0.1), (2, 0.2), (3, 0.3)):                         # subset form: b' = max(int(b(1-r)),1) kept at b/b'
        for key in ("rs1", "rs2"):
            r = blocks[i][key]
            bsub = max(int(Bc * (1.0 - m.dpr[i])), 1)
            assert int((r > 0).sum()) == bsub
            assert torch.allclose(r[r > 0], torch.full((bsub,), Bc / bsub, device=dev))
    assert not torch.equal(blocks[3]["rs1"], blocks[3]["rs2"])             # independent draws per branch
    # per-sample DropPath (rates <= 0.1): scales are bernoulli(keep) / keep
    m2 = DinoVisionTransformer(img_size=32, patch_size=16, embed_dim=128, depth=3, num_heads=2, init_values=1.0,
                               drop_path_rate=0.08, requires_grad=True)
    c2 = m2._fwd(x, None, save=True, drop_path=True)
    for i in (1, 2):
        vals = set(round(v, 4) for v in c2.blocks[i]["rs1"].tolist())
        assert vals <= {0.0, round(1 / (1 - m2.dpr[i]), 4)} and len(vals) >= 1
    # gradient isolation: cotangent only on sample j's tokens; a block-3 branch dropped for sample j must not see it
    N = ctx.dims[3]
    j = int((blocks[3]["rs2"] == 0).nonzero()[0])
    d = torch.zeros(Bc * N, 128, device=dev)
    d[j * N:(j + 1) * N] = torch.randn(N, 128, device=dev)
    g0 = m.arena.g("blocks.3.mlp.fc2.weight")
    m._bwd(ctx, d)
    torch.cuda.synchronize()
    assert g0.abs().max().item() == 0.0, "dropped sample leaked gradient into its dropped MLP branch"
    assert m.arena.g("blocks.0.mlp.fc2.weight").abs().max().item() > 0.0


@pytest.mark.parametrize("ckpt", [False, True])
def test_subset_stochastic_depth_compact_equals_dense(ckpt):
    """Batch-subset stochastic depth (layers/block.py:118-141): the compact schedule (only the kept samples go through the
    branch: gather -> branch -> scaled write-back) must reproduce the dense statement (every sample computed, dropped ones
    multiplied by zero) for the same random subsets -- forward features and every parameter gradient."""
    Bc = 16
    x = torch.randn(Bc, 3, 64, 64, device=dev)

    def run(compact: bool):
        torch.manual_seed(5)
        m = DinoVisionTransformer(img_size=64, patch_size=16, embed_dim=128, depth=3, num_heads=2, init_values=0.7,
                                  drop_path_rate=0.3, drop_path_uniform=True, requires_grad=True)
        m.subset_skips_compute = compact
        m._activation_checkpointing = ckpt
        m.arena.zero_grad()
        torch.manual_seed(11)  # same subset draws in both schedules
        ctx = m._fwd(x, None, save=True, drop_path=True)
        out = ctx.xnorm.clone()
        kept = [int((blk["rs1"] > 0).sum()) for blk in ctx.blocks] if compact else None
        cot = torch.randn(out.shape, generator=torch.Generator().manual_seed(9)).to(dev)
        m._bwd(ctx, cot)
        torch.cuda.synchronize()
        return out, m.arena.grad.clone(), kept

    o_d, g_d, _ = run(False)
    o_c, g_c, kept = run(True)
    assert kept == [max(int(Bc * 0.7), 1)] * 3
    assert (o_d - o_c).abs().max().item() < 2e-2 and (o_d - o_c).abs().mean().item() < 1e-3  # same math, bf16 tiles regrouped
    assert ((g_d - g_c).norm() / g_d.norm()).item() < 2e-2


def test_cut_backbone_backward_equals_uncut():
    """The backbone backward cut between blocks (the second all-reduce bucket boundary of multi-GPU runs) must produce the same
    gradients as the uncut schedule -- eager and graph replay."""
    from tests.golden import recipes as Rr
    import oracle.dinov2_oracle as Oo
    vit = Oo.ViTConfig(embed_dim=128, depth=4, num_heads=2, patch_size=16, img_size=224, init_values=1e-5)
    cfg = Oo.StepConfig(vit=vit, head=Rr.HEAD_TINY)
    st = Rr.det_step_state(cfg, seed=43)
    views, masks, idx, w = Rr.step_case_inputs(cfg)
    batch = {"views": [v.to(dev) for v in views], "masks": {"collated_masks": masks, "mask_indices_list": idx, "masks_weight": w}}

    def run(split, graph):
        margs = DINOv2Args(hidden_dim=cfg.head.hidden_dim, dino_bottleneck_dim=cfg.head.bottleneck_dim, output_dim=cfg.head.out_dim)
        mk = dict(img_size=224, patch_size=16, embed_dim=128, depth=4, num_heads=2, init_values=1e-5, drop_path_rate=0.0)
        m = DINOv2(margs, DINOv2AdamWViTArgs(), mk, 1024, 3, max_steps=10, device=dev)
        m.s_arena.load_from(st["student"]); m.t_arena.load_from(st["teacher"])
        m.force_backbone_split = split
        res = m._graphed_step(batch) if graph else m.training_step_impl(batch, 0)
        torch.cuda.synchronize()
        return float(res.loss), m.s_arena.grad.clone()

    l0, g0 = run(0, False)
    for split, graph in ((2, False), (2, True), (1, True)):
        l1, g1 = run(split, graph)
        assert abs(l0 - l1) < 1e-5 * abs(l0)
        assert (g0 - g1).abs().max().item() < 2e-4 * g0.abs().max().item(), (split, graph)
