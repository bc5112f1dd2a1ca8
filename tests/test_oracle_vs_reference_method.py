"""CPU: the oracle's training step pinned against the reference's OWN method class (`DINOv2.training_step_impl` and its
optimizer / EMA hooks, unmodified source, run through oracle/ref_full.py by tools/make_method_golden.py, which stored
its loss terms, gradients and post-step weights under tests/golden/) on identical weights, crops and masks.

This pins what the module-level fixtures cannot: the glue of dinov2.py:259-397 (crop order, A<->B swap, loss scaling),
configure_optimizers' param groups, and the hook ORDER of one optimisation step (weight-decay schedule and lr freeze at
global_step, EMA momentum at global_step + 1 because Lightning increments before on_train_batch_end).
Gradients and weights are compared norm-wise and at the elements of `recipes.sample_index` the fixture keeps."""
import pytest
import torch

from oracle import dinov2_oracle as O
from tests import ref_cases as RC
from tests.golden import recipes as R


@pytest.mark.parametrize("case", [RC.TINY, RC.TINY_SK], ids=lambda c: c.name)
def test_oracle_step_matches_reference_method(case, golden_dir):
    torch.set_num_threads(8)
    ref = torch.load(golden_dir / f"method_step_{case.name}.pt")
    terms = ref["terms"]
    views = RC.make_views(case)
    cfg = RC.oracle_cfg(case)
    st = R.det_step_state(cfg, seed=41)
    teacher, centers = st["teacher"], st["centers"]
    student = {k: v.clone().requires_grad_(True) for k, v in st["student"].items()}
    assert list(student) == ref["names"]
    mk = RC.masks_for(case, 11)
    out = O.training_step(cfg, student, teacher, centers, views, mk["collated_masks"], mk["mask_indices_list"],
                          mk["masks_weight"], teacher_temp=0.05)
    for k in ("loss", "dino_global_loss", "dino_local_loss", "ibot_loss", "koleo_loss"):
        assert abs(float(out[k]) - terms[k]) < 2e-5 * max(1.0, abs(terms[k])), (k, float(out[k]), terms[k])
    out["loss"].backward()
    idx = {k: R.sample_index(p.numel(), ref["grad_sample"].shape[1]) for k, p in student.items()}
    worst = 0.0
    for i, (k, p) in enumerate(student.items()):
        gnorm = float(ref["grad_norm"][i])
        # relative error of the sampled elements, scaled to the whole tensor's norm (an estimate of |g - g_ref| / |g_ref|)
        scale = (p.numel() / idx[k].numel()) ** 0.5
        e = (p.grad.flatten()[idx[k]] - ref["grad_sample"][i]).norm().item() * scale / (gnorm + 1e-12)
        worst = max(worst, e, abs(p.grad.norm().item() - gnorm) / (gnorm + 1e-12))
    assert worst < 1e-4, worst

    # ---- one full optimisation step of the reference in Lightning's hook order vs the oracle's optimizer restatement
    a = ref["args"]
    p = {k: v.detach().clone() for k, v in student.items()}
    g = [student[k].grad.detach().clone() for k in p]
    O.clip_grad_norm(g, a["gradient_clip_val"])
    base_lr = 0.004 * (case.batch / 1024) ** 0.5
    lr = base_lr * O.cosine_warmup_lr_factor(0, 2, 10, a["min_lr"] / base_lr)
    wd_now = O.cosine_schedule(0, 10, 0.04, a["weight_decay_end"])
    for (k, pk), gk in zip(p.items(), g):
        is_bb = k.startswith("backbone.")
        hp = O.param_hparams(k[len("backbone."):] if is_bb else k, is_bb, lr, 1.0, cfg.vit.depth)
        lr_k = 0.0 if "last_layer" in k else hp["lr"]  # student_freeze_last_layer_steps=1: frozen at step 0
        O.adamw_step(pk, gk, torch.zeros_like(pk), torch.zeros_like(pk), 1, lr_k, wd_now * hp["weight_decay"])
    mom = O.cosine_schedule(1, 10, a["momentum_start"], a["momentum_end"])  # global_step + 1
    t = {k: v.clone() for k, v in teacher.items()}
    O.update_ema([p[k] for k in p], [t[k] for k in p], mom)

    def close(x, y, what, gr):
        # e.g. the k-third of qkv.bias: its gradient is exactly zero in exact arithmetic
        keep = gr.abs() > 1e-6 * gr.abs().max()
        x, y = x[keep], y[keep]
        # Adam's first step is lr * g/|g|: elements whose gradient is at rounding-noise level can land anywhere in
        # +-lr (1.1e-4 here), so a handful of outliers well below lr are tolerated; everything else must agree to 2e-5
        bad = (x - y).abs() > 1e-6 + 2e-5 * y.abs()
        assert int(bad.sum()) <= max(3, int(5e-4 * bad.numel())) and (x - y).abs().max().item() < 2e-5, (what, int(bad.sum()), (x - y).abs().max().item())

    for i, k in enumerate(p):
        gr = student[k].grad.flatten()[idx[k]]
        close(p[k].flatten()[idx[k]], ref["student_after"][i], "student " + k, gr)
        close(t[k].flatten()[idx[k]], ref["teacher_after"][i], "teacher " + k, gr)
    # a momentum taken at global_step (one step early) would be visibly different
    mom_early = O.cosine_schedule(0, 10, a["momentum_start"], a["momentum_end"])
    assert abs(mom - mom_early) > 1e-5
