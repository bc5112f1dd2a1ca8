#!/usr/bin/env python
"""bench.py -- images/sec of the full DINOv2 training step (default cfg2: ViT-S/16, 2x224^2 + 8x96^2 crops, bs 64/GPU).

    python bench.py --gpus N --steps K --warmup W            # B200 arm (this repo's kernels)
    python bench.py --impl reference --steps K --warmup W     # reference arm: the reference's own method class on host cores
    python bench.py --config cfg3|cfg5 ...                    # BASELINE.json configs[2] / configs[4] (headline stays cfg2)

One "step" = teacher forward, student forward+backward (global + local crops), DINO/iBOT/KoLeo losses,
gradient all-reduce (N>1), clip + AdamW + EMA teacher.  Synthetic N(0,1) crops, random-init weights.
`value`  : whole-job images/s with inputs resident in HBM when the timed region starts.
`e2e`    : the same step through the public API with HOST (pinned) crops: H2D copy of every step's views and
           a D2H read of every step's loss inside the timed region (double-buffered on a copy stream).
`roofline`: tcgen05 GEMM launches of one step timed with CUDA events on the launch stream (raw event time, no
           subtraction); `rooflines_hbm`: the loss kernels (row_lse + dino_ce) and the fused optimizer sweep against the
           measured HBM copy bandwidth, timed the same way in the same step.
`parity` : one step of the bench model (same weights, drop-path off) on the first 4 images of the bench batch against
           the autocast-emulating oracle on the host: loss delta and logit errors.
`cpu_baseline` / `--impl reference`: the reference's OWN DINOv2 method class (unmodified source from baseline/_ref or
           $LIGHTLY_TRAIN_SRC, absent third-party packages stubbed: oracle/ref_full.py) on the host cores;
`gpu_torch_baseline`: those same reference modules on the B200 under torch.autocast(bf16), eager -- "the kernel to beat".
`--dump-outputs DIR`: after the timed steps, what the last of them handed back (loss and its terms) and left in the model
           (a fixed, seeded sample of the student / teacher weights, the loss centers) as DIR/<name>.npy, so that two
           builds can be compared output for output on identical inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

# BASELINE.json `configs`: [1] is the headline the metric is quoted on; [2] and [4] are extra workloads
CONFIGS = {
    "cfg2": dict(
        vit=dict(img_size=224, patch_size=16, embed_dim=384, depth=12, num_heads=6, init_values=1e-5, drop_path_rate=0.1),
        method={}, batch=64, n_local=8, local=96, ckpt=False,
        metric="images/sec ViT-S/16 DINOv2 training step (2g+8l crops, bs64/GPU)",
        workload="cfg2: ViT-S/16 DINOv2, 2x224^2 + 8x96^2 crops, bs=%d/GPU, K=65536 shared DINO/iBOT head, softmax centering, "
                 "drop_path 0.1, full step incl. clip+AdamW+EMA"),
    "cfg3": dict(
        vit=dict(img_size=224, patch_size=14, embed_dim=768, depth=12, num_heads=12, init_values=1e-5, drop_path_rate=0.2,
                 ffn_layer="swiglufused", num_register_tokens=4, interpolate_antialias=True, interpolate_offset=0.0),
        method=dict(ibot_separate_head=True, center_method="sinkhorn_knopp"), batch=32, n_local=8, local=98, ckpt=False,
        metric="images/sec ViT-B/14 reg4 DINOv2 training step (iBOT head + Sinkhorn-Knopp, 2g+8l crops, bs32/GPU)",
        workload="cfg3: ViT-B/14 reg4 SwiGLU DINOv2, 2x224^2 + 8x98^2 crops, bs=%d/GPU, K=65536 separate DINO and iBOT heads, "
                 "Sinkhorn-Knopp centering, drop_path 0.2, full step incl. clip+AdamW+EMA"),
    "cfg5": dict(
        vit=dict(img_size=224, patch_size=16, embed_dim=1024, depth=24, num_heads=16, init_values=1e-5, drop_path_rate=0.3,
                 drop_path_uniform=True),
        method={}, batch=16, n_local=10, local=96, ckpt=True,
        metric="images/sec ViT-L/16 DINOv2 training step (2g+10l crops, bs16/GPU, activation checkpointing)",
        workload="cfg5: ViT-L/16 DINOv2, 2x224^2 + 10x96^2 crops, bs=%d/GPU, K=65536 shared head, softmax centering, "
                 "drop_path 0.3 uniform (batch-subset form), activation checkpointing on, full step incl. clip+AdamW+EMA"),
    "cfg4": dict(
        batch=128,
        metric="images/sec DistillationV3 step (DINOv3 ViT-B/16 teacher -> ResNet-50 student, 224^2, bs128/GPU)",
        workload="cfg4: distillation, DINOv3 ViT-B/16 teacher (RoPE, 4 storage tokens; this repo's sm_100a kernels, forward only) -> "
                 "torchvision ResNet-50 student (cuDNN via torch.autograd, channels-last bf16 autocast), one 224^2 view, bs=%d/GPU, "
                 "queue 8192, fused KL kernels, full step incl. student backward + AdamW"),
}


def make_views(batch: int, n_local: int, seed: int, device, pin: bool = False, local: int = 96):
    g = torch.Generator().manual_seed(seed)
    views = [torch.randn(batch, 3, 224, 224, generator=g) for _ in range(2)]
    views += [torch.randn(batch, 3, local, local, generator=g) for _ in range(n_local)]
    if device is not None:
        return [v.to(device) for v in views]
    if pin:
        return [v.pin_memory() for v in views]
    return views


def _bind_to_gpu_cores(local_rank: int):
    """Restrict this process to the CPU cores NVML reports as local to GPU `local_rank`; returns the previous affinity (or
    None when the topology cannot be read: nothing is changed then)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        n = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cpus = {i for i in range(n) if (words[i // 64] >> (i % 64)) & 1}
        old = os.sched_getaffinity(0)
        cpus &= old
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return old
    except Exception:
        return None


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    def __init__(self, index: int) -> None:
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._idx = index
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self) -> None:
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self._idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=5)

    def summary(self) -> dict:
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# --------------------------------------------------------------------------------------------- reference on the host / GPU
def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def _ref_case(cfg: dict, batch: int):
    from tests import ref_cases as RC

    vit = dict(cfg["vit"])
    vit.setdefault("mlp_ratio", 4)
    vit["block_chunks"] = 0
    return RC.Case("bench", vit, method=dict(cfg["method"]), batch=batch, n_local=cfg["n_local"], local_size=cfg["local"],
                   checkpointing=cfg["ckpt"])


def reference_step_time(cfg: dict, batch: int, steps: int, warmup: int, threads: int, device: str = "cpu"):
    """Seconds per full optimisation step of the reference's own DINOv2 method class (training_step_impl + backward +
    its optimizer / clipping / EMA hooks in Lightning's order).  device="cuda": under torch.autocast(bf16), CUDA events."""
    from oracle import ref_full
    import random

    if device == "cpu":
        torch.set_num_threads(threads)
    case = _ref_case(cfg, batch)
    torch.manual_seed(0)
    m, opt, sched = ref_full.build_dinov2(case.vit, dict(case.method), global_batch_size=batch, max_steps=125_000, device=device,
                                          activation_checkpointing=case.checkpointing)
    views = make_views(batch, cfg["n_local"], 123, None if device == "cpu" else device, local=cfg["local"])
    random.seed(0)
    times = []
    for it in range(warmup + steps):
        if device == "cpu":
            t0 = time.perf_counter()
            ref_full.run_step(m, opt, sched, {"views": views})
            dt = time.perf_counter() - t0
        else:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ref_full.run_step(m, opt, sched, {"views": views}, autocast_device="cuda")
            e1.record()
            torch.cuda.synchronize()
            dt = e0.elapsed_time(e1) / 1e3
        if it >= warmup:
            times.append(dt)
    return sum(times) / len(times)


def port_step_time(batch: int, steps: int, warmup: int, threads: int):
    """Fallback when no reference copy is on the box: the oracle port of the same step (fwd, autograd bwd, clip, AdamW, EMA)."""
    from oracle import dinov2_oracle as O
    from tests.golden import recipes as R

    torch.set_num_threads(threads)
    vit = O.ViTConfig(embed_dim=384, depth=12, num_heads=6, patch_size=16, img_size=224, init_values=1e-5)
    head = O.HeadConfig(in_dim=384, hidden_dim=2048, bottleneck_dim=256, out_dim=65536)
    cfg = O.StepConfig(vit=vit, head=head)
    st = R.det_step_state(cfg, seed=7)
    student = {k: v.clone().requires_grad_(True) for k, v in st["student"].items()}
    teacher = st["teacher"]
    m_state = {k: torch.zeros_like(v) for k, v in student.items()}
    v_state = {k: torch.zeros_like(v) for k, v in student.items()}
    views = make_views(batch, 8, 123, None)
    g = torch.Generator().manual_seed(5)
    masks = torch.rand(2 * batch, 196, generator=g) < 0.15
    masks[batch:] = False
    idx = masks.flatten().nonzero().flatten()
    w = O.masks_weight_from_masks(masks)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        for p in student.values():
            p.grad = None
        out = O.training_step(cfg, student, teacher, st["centers"], views, masks, idx, w, teacher_temp=0.04)
        out["loss"].backward()
        with torch.no_grad():
            grads = [p.grad for p in student.values()]
            O.clip_grad_norm(grads, 3.0)
            for k, p in student.items():
                hp = O.param_hparams(k[len("backbone."):] if k.startswith("backbone.") else k, k.startswith("backbone."),
                                     1e-3, 0.04, 12)
                O.adamw_step(p, p.grad, m_state[k], v_state[k], it + 1, hp["lr"], hp["weight_decay"])
            O.update_ema(list(student.values()), [teacher[k] for k in student], 0.992)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return sum(times) / len(times)


def cpu_reference(cfg: dict, steps: int, warmup: int, sweep: bool):
    """(images/s, description dict) of the reference on the host cores: its own method class when a copy of the
    reference is on the box (kind "reference"), else the oracle port (kind "port")."""
    from oracle import ref_full

    cores = host_cores()
    if not ref_full.available():
        threads = min(cores, 16)
        sec = port_step_time(4, steps, warmup, threads)
        return 4 / sec, {"kind": "port", "cores": threads, "batch": 4,
                         "sample": "full step at bs=4 (reference algorithm restated in oracle/, torch CPU fp32); no reference copy on this box"}
    best = None
    tried = []
    cands = [(t, b) for t in (16, 32, 64) if t <= cores for b in (4, 8)] if sweep else [(min(cores, 32), 4)]
    if not cands:
        cands = [(cores, 4)]
    for threads, batch in cands:
        sec = reference_step_time(cfg, batch, 1, 1, threads)
        tried.append({"threads": threads, "batch": batch, "images_per_s": round(batch / sec, 3)})
        if best is None or batch / sec > best[0]:
            best = (batch / sec, threads, batch)
    _, threads, batch = best
    sec = reference_step_time(cfg, batch, steps, warmup, threads)
    return batch / sec, {"kind": "reference", "cores": threads, "batch": batch, "host_cores": cores, "sweep": tried,
                         "sample": f"the reference's own DINOv2 method class (training_step_impl + backward + optimizer/clip/EMA hooks; "
                                   f"source: {ref_full.source_root()}, pytorch_lightning/lightly stubbed by oracle/ref_full.py), torch CPU fp32, "
                                   f"bs={batch} per step (a bounded sample of the bs-64 workload), {threads} threads"}


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    if "vit" not in cfg:
        print(json.dumps({"impl": "reference", "unavailable": f"no host reference arm for {args.config} (only the DINOv2 configs)"}), flush=True)
        return
    value, desc = cpu_reference(cfg, args.steps, args.warmup, sweep=True)
    batch = desc["batch"]
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": value,
        "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": batch / value * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": cfg["workload"] % cfg["batch"],
                   "global_batch": cfg["batch"] * args.gpus, "parallelism": f"dp{args.gpus}",
                   "measured_on": f"host CPU, fp32, {desc['cores']} threads, bs={batch} per step: a bounded sample of the workload "
                                  "(the B200 arm runs the full per-GPU batch in bf16); one host regardless of --gpus"},
        "cpu_baseline": {"value": value, "unit": "images/s", **desc},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- output dump
DUMP_SAMPLE = 1 << 20  # elements kept of each large tensor (4 MB in float32)


def _sample(x: "torch.Tensor", seed: int) -> "torch.Tensor":
    """A fixed, seeded sample of DUMP_SAMPLE elements of a flat tensor (all of it when smaller)."""
    x = x.detach().flatten()
    if x.numel() <= DUMP_SAMPLE:
        return x
    idx = torch.randint(0, x.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(seed)).to(x.device)
    return x[idx]


def dump_outputs(out_dir: str, res, tensors: dict) -> None:
    """Write the step result (loss and every log_dict term) and `tensors` (sampled) as float32 .npy files."""
    import numpy as np

    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    arrays = {"loss": res.loss}
    arrays.update({k.split("/")[-1]: v for k, v in res.log_dict.items()})
    arrays.update({k: _sample(v, seed=i) for i, (k, v) in enumerate(tensors.items())})
    for k, v in arrays.items():
        np.save(d / f"{k}.npy", torch.as_tensor(v).detach().float().cpu().numpy())


# --------------------------------------------------------------------------------------------- parity of the bench model
def bench_parity(method, cfg: dict, views_dev, dev) -> dict:
    """One step (drop-path off, eager) of a copy of the bench model on the first 4 images of the bench batch vs the
    autocast-emulating oracle on the host: |loss delta| and logit errors (north_star: 1e-3 on logits / loss)."""
    import random

    from lightly_train_b200._methods.dinov2.dinov2 import DINOv2, DINOv2AdamWViTArgs, DINOv2Args
    from oracle import dinov2_oracle as O
    from tests import ref_cases as RC

    nb = 4
    vit = dict(cfg["vit"]); vit["drop_path_rate"] = 0.0; vit.pop("drop_path_uniform", None)
    margs = dict(cfg["method"]); margs.update(teacher_temp_start=0.05, teacher_temp_end=0.05)
    m = DINOv2(DINOv2Args(**margs), DINOv2AdamWViTArgs(), vit, nb, 3, max_steps=100, device=str(dev))
    m.s_arena.fp32.copy_(method.s_arena.fp32); m.t_arena.fp32.copy_(method.t_arena.fp32)
    m.s_arena.bf16_valid = m.t_arena.bf16_valid = False
    method.dino_loss.apply_center_update(); method.ibot_loss.apply_center_update()
    m.dino_loss.center.copy_(method.dino_loss.center); m.ibot_loss.center.copy_(method.ibot_loss.center)
    views = [v[:nb].contiguous() for v in views_dev]
    case = RC.Case("bench", dict(vit, block_chunks=0, mlp_ratio=4), method=dict(cfg["method"]), batch=nb, n_local=cfg["n_local"],
                   local_size=cfg["local"])
    mk = RC.masks_for(case, 17)
    m.debug_taps = {}
    res = m.training_step_impl({"views": views, "masks": mk}, 0)
    torch.cuda.synchronize()
    student = {k: m.s_arena.p(k).detach().cpu().clone() for k in m.s_arena.names()}
    teacher = {k: m.t_arena.p(k).detach().cpu().clone() for k in m.t_arena.names()}
    centers = {"dino": m.dino_loss.center.cpu().clone(), "ibot": m.ibot_loss.center.cpu().clone()}
    taps = {}
    torch.set_num_threads(min(host_cores(), 32))
    with torch.no_grad():
        out = O.training_step(RC.oracle_cfg(case), student, teacher, centers, [v.cpu() for v in views], mk["collated_masks"],
                              mk["mask_indices_list"], mk["masks_weight"], teacher_temp=0.05, autocast=True, taps=taps)
    want_t = torch.cat([taps["t_cls_logits"], taps["t_patch_logits"]])
    want_s = torch.cat([taps["s_cls_logits_g"]] + ([taps["s_cls_logits_l"]] if cfg["n_local"] else []) + [taps["s_patch_logits"]])
    dt = (m.debug_taps["t_logits"].float().cpu() - want_t).abs()
    ds = (m.debug_taps["s_logits"].float().cpu() - want_s).abs()
    return {"against": "oracle (autocast-emulating CPU restatement of the reference step), first 4 images of the bench batch, "
                       "bench weights, drop-path off, teacher_temp 0.05",
            "loss_cuda": float(res.loss), "loss_oracle": float(out["loss"]),
            "loss_delta_vs_oracle": abs(float(res.loss) - float(out["loss"])),
            "term_deltas": {k.split("/")[1]: abs(float(v) - float(out[k.split("/")[1]])) for k, v in res.log_dict.items()},
            "max_logit_err": max(dt.max().item(), ds.max().item()), "mean_logit_err": 0.5 * (dt.mean().item() + ds.mean().item()),
            "logit_rows": int(dt.shape[0] + ds.shape[0])}


# --------------------------------------------------------------------------------------------- cfg4: distillation
def run_distill(args) -> None:
    """BASELINE.json configs[3].  The teacher forward (the ViT-B FLOPs) and the loss run on this repo's kernels; the
    convolutional student, its backward and its AdamW are torch / cuDNN (library code, stated in the workload string)."""
    import torch.distributed as dist
    import torchvision

    from lightly_train_b200 import _lib, ops
    from lightly_train_b200._methods.distillationv3.distillationv3 import DistillationV3, DistillationV3Args
    from lightly_train_b200._models.dinov3_vit import DinoV3VisionTransformer, DINOv3ViTModelWrapper
    from lightly_train_b200._models.torchvision_resnet import EmbeddingModel, ResNetModelWrapper

    cfg = CONFIGS["cfg4"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    W, K, B = max(args.warmup, 3), args.steps, args.batch or cfg["batch"]
    torch.manual_seed(0)
    teacher = DinoV3VisionTransformer(img_size=224, patch_size=16, embed_dim=768, depth=12, num_heads=12, ffn_ratio=4.0,
                                      layerscale_init=1e-5, norm_layer="layernormbf16", n_storage_tokens=4, mask_k_bias=True,
                                      pos_embed_rope_dtype="fp32", device=str(dev))
    student = EmbeddingModel(ResNetModelWrapper(torchvision.models.resnet50())).to(dev).to(memory_format=torch.channels_last)
    method = DistillationV3(DistillationV3Args(), None, student, B * world, 3,
                            teacher_embedding_model=DINOv3ViTModelWrapper(teacher)).to(dev)
    params = [p for p in method.parameters() if p.requires_grad]
    if world > 1:
        for p in params:
            dist.broadcast(p.data, 0)
    opt = torch.optim.AdamW(params, lr=5e-4, weight_decay=0.04, fused=True)
    g = torch.Generator().manual_seed(1000 + rank)
    batches = [torch.randn(B, 3, 224, 224, generator=g).to(dev).contiguous(memory_format=torch.channels_last) for _ in range(2)]

    def step(x):
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            res = method.training_step_impl({"views": [x]}, 0)
        res.loss.backward()
        if world > 1:
            for p in params:
                dist.all_reduce(p.grad)
                p.grad.div_(world)
        opt.step()
        return res

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(W):
        step(batches[i % 2])
    barrier()
    l0 = _lib.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        barrier()
        e0.record()
        for i in range(K):
            res = step(batches[i % 2])
        e1.record()
        barrier()
    launches = _lib.LAUNCHES - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, {"student_params": torch.cat([p.detach().flatten() for p in params])})
    t = torch.tensor([e0.elapsed_time(e1) / K], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    # e2e: pinned host images -> device every step, loss read back every step
    host = [torch.randn(B, 3, 224, 224, generator=g).pin_memory() for _ in range(2)]
    dbuf = [torch.empty(B, 3, 224, 224, device=dev).contiguous(memory_format=torch.channels_last) for _ in range(2)]
    lh = torch.zeros(1).pin_memory()

    def e2e_run(n):
        for i in range(n):
            dbuf[i % 2].copy_(host[i % 2], non_blocking=True)
            r = step(dbuf[i % 2])
            lh.copy_(r.loss.detach().reshape(1), non_blocking=True)
        torch.cuda.synchronize()

    e2e_run(2)
    barrier()
    e0.record(); e2e_run(K); e1.record()
    barrier()
    t2 = torch.tensor([e0.elapsed_time(e1) / K], device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    # roofline: the teacher's tcgen05 GEMMs of one step, CUDA events per launch
    ops.GEMM_PROFILE = []
    step(batches[0])
    torch.cuda.synchronize()
    prof, ops.GEMM_PROFILE = ops.GEMM_PROFILE, None
    peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
    if rank == 0:
        flops = sum(f for f, _, _ in prof)
        gms = sum(a.elapsed_time(b) for _, a, b in prof)
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        line = {"metric": cfg["metric"], "value": B * world / (ms / 1e3), "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": cfg["workload"] % B, "global_batch": B * world, "parallelism": f"dp{world}",
                           "l2_policy": "2 alternating 77 MB input batches; activations exceed the 126 MB L2"},
                "clocks": clk.summary(),
                "e2e": {"value": B * world / (float(t2[0]) / 1e3), "unit": "images/s", "h2d_bytes_per_step": B * 3 * 224 * 224 * 4,
                        "d2h_bytes_per_step": 4},
                "gpu_launches": launches, "gpu_launches_scope": "library (libb200dino.so) kernel launches of rank 0: teacher + loss; the student's cuDNN / ATen launches are not counted",
                "loss": float(res.loss),
                "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (teacher forward, all launches of one step)",
                             "achieved": flops / (gms * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s", "frac": flops / (gms * 1e-3) / 1e12 / peak,
                             "traffic": None, "gemm_launches": len(prof), "gemm_ms_per_step": gms,
                             "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained"},
                "cpu_baseline": None}
        if os.environ.get("B200_BENCH_DIAG_NO_ALLREDUCE", "0") == "1":
            line["diagnostic"] = "gradient all-reduce DISABLED (B200_BENCH_DIAG_NO_ALLREDUCE=1): not a training step, not a bench value"
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------- B200 arm
def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--eager", action="store_true", help="launch every kernel from the host instead of CUDA-graph replay")
    ap.add_argument("--gemm-profile", default="", help="write the per-shape GEMM timing table of one step to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32, large tensors sampled)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.config == "cfg4":
        run_distill(args)
        return

    import torch.distributed as dist

    from lightly_train_b200 import _lib, ops
    from lightly_train_b200._methods.dinov2.dinov2 import DINOv2, DINOv2AdamWViTArgs, DINOv2Args

    cfg = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's version banner must not precede the JSON line on stdout
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    W = max(args.warmup, 3)
    K = args.steps
    B = args.batch or cfg["batch"]
    NL, LS = cfg["n_local"], cfg["local"]

    import random
    random.seed(1000 + rank)
    torch.manual_seed(0)
    method = DINOv2(DINOv2Args(**cfg["method"]), DINOv2AdamWViTArgs(), dict(cfg["vit"]), B * world, 3, max_steps=125_000, device=str(dev))
    if cfg["ckpt"]:
        method.student_embedding_model.wrapped_model.set_activation_checkpointing(True)
    method.use_cuda_graph = not args.eager
    diag = os.environ.get("B200_BENCH_DIAG_NO_ALLREDUCE", "0") == "1"
    if diag:  # DIAGNOSTIC ONLY (line is flagged): the step without its gradient all-reduce = the ceiling of overlap tuning
        method._allreduce_head_grads_async = lambda: None
        method._allreduce_upper_backbone_async = lambda split_at: None
        method._finish_grad_allreduce = lambda: None
    if world > 1:  # identical initial weights on every rank
        dist.broadcast(method.s_arena.fp32, 0)
        dist.broadcast(method.t_arena.fp32, 0)
        method.s_arena.bf16_valid = method.t_arena.bf16_valid = False
    # two distinct resident batches (134 MB each at cfg2, larger than L2) alternate between steps
    batches = [{"views": make_views(B, NL, 1000 * rank + i, dev, local=LS)} for i in range(2)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(W):
        method.train_step(batches[i % 2])
    barrier()
    l0 = _lib.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        barrier()
        e0.record()
        h0 = time.perf_counter()
        for i in range(K):
            res = method.train_step(batches[i % 2])
        host_ms = (time.perf_counter() - h0) / K * 1e3  # host time to enqueue one step (must stay below ms_per_step)
        e1.record()
        barrier()
    launches = _lib.LAUNCHES - l0
    ms = e0.elapsed_time(e1) / K
    loss_val = float(res.loss)
    if args.dump_outputs and rank == 0:  # before the e2e steps below overwrite the graph's outputs and the weights
        dump_outputs(args.dump_outputs, res, {"student_params": method.s_arena.fp32, "teacher_params": method.t_arena.fp32,
                                              "dino_center": method.dino_loss.center, "ibot_center": method.ibot_loss.center})
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    value = B * world / (ms / 1e3)

    # ---- e2e: host (pinned) crops -> device every step on a copy stream, loss read back every step
    e2e = None
    if not args.no_e2e:
        # the pinned staging buffers are allocated (first-touched) from the CPU cores that are local to this rank's GPU, as a
        # launcher would with numactl: with several ranks per host every rank otherwise pins its buffers wherever it happens
        # to run (B200_BENCH_NUMA_BIND=0 disables; the previous affinity is restored right after the allocation)
        old_aff = _bind_to_gpu_cores(local_rank) if os.environ.get("B200_BENCH_NUMA_BIND", "0") == "1" else None
        host = [make_views(B, NL, 2000 * rank + i, None, pin=True, local=LS) for i in range(2)]
        if old_aff is not None:
            os.sched_setaffinity(0, old_aff)
        h2d_bytes = sum(v.numel() * 4 for v in host[0])
        copy_stream = torch.cuda.Stream(device=dev)
        dev_bufs = [[torch.empty_like(v, device=dev) for v in host[0]] for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        loss_host = torch.zeros(2).pin_memory()
        loss_done = [torch.cuda.Event() for _ in range(2)]
        losses: list = []

        def prefetch(i: int) -> None:
            slot = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])
                for d, h in zip(dev_bufs[slot], host[slot]):
                    d.copy_(h, non_blocking=True)
                ready[slot].record(copy_stream)

        def run_e2e(n: int) -> None:
            for s in range(2):
                consumed[s].record(torch.cuda.current_stream())
            prefetch(0)
            for i in range(n):
                slot = i % 2
                if i + 1 < n:
                    prefetch(i + 1)
                torch.cuda.current_stream().wait_event(ready[slot])
                r = method.train_step({"views": dev_bufs[slot]})
                consumed[slot].record(torch.cuda.current_stream())
                # D2H of every step's loss into pinned memory; the host waits for it one step later (after the next
                # step has been enqueued), as a logging trainer does, so the device never idles on the read-back
                loss_host[slot:slot + 1].copy_(r.loss.reshape(1), non_blocking=True)
                loss_done[slot].record(torch.cuda.current_stream())
                if i >= 1:
                    loss_done[1 - slot].synchronize()
                    losses.append(float(loss_host[1 - slot]))
            loss_done[(n - 1) % 2].synchronize()
            losses.append(float(loss_host[(n - 1) % 2]))

        run_e2e(2)
        barrier()
        e0.record()
        run_e2e(K)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) / K], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": B * world / (float(t[0]) / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": 4}

    # ---- rooflines: every tcgen05 GEMM launch, the loss kernels and the optimizer sweep of one eagerly launched step,
    # each bracketed by a CUDA-event pair on the launch stream (every rank runs the step: it contains the all-reduce)
    roofline = None
    rooflines_hbm = None
    ops.GEMM_PROFILE = []
    ops.KERNEL_PROFILE = []
    method.use_cuda_graph = False  # events cannot be recorded inside a graph replay: time the eager schedule
    torch.cuda._sleep(int(3e8))    # ~150 ms head start for the host, so event pairs bracket kernels, not launch gaps
    method.train_step(batches[0])
    torch.cuda.synchronize()
    method.use_cuda_graph = not args.eager
    prof, ops.GEMM_PROFILE = ops.GEMM_PROFILE, None
    kprof, ops.KERNEL_PROFILE = ops.KERNEL_PROFILE, None
    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    if rank == 0:
        if args.gemm_profile:
            table = {}
            for (f, a, b), key in zip(prof, ops.GEMM_PROFILE_KEYS):
                tt = table.setdefault(key, [0, 0.0, 0.0])
                tt[0] += 1; tt[1] += a.elapsed_time(b); tt[2] += f
            rows = sorted(((k, v) for k, v in table.items()), key=lambda kv: -kv[1][1])
            with open(args.gemm_profile, "w") as fh:
                fh.write("M,N,K,a_mn,b_mn,epi,splits,launches,total_ms,TFLOP/s\n")
                for k, v in rows:
                    fh.write(",".join(map(str, k)) + f",{v[0]},{v[1]:.4f},{v[2] / (v[1] * 1e-3) / 1e12:.1f}\n")
        flops = sum(f for f, _, _ in prof)
        gemm_ms = sum(a.elapsed_time(b) for _, a, b in prof)
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        ach = flops / (gemm_ms * 1e-3) / 1e12
        traffic = None
        tf = ROOT / "profiles" / "r02_gemm_traffic.json"  # dram bytes per launch from this round's `ncu --set full` capture
        if tf.exists() and args.config == "cfg2" and B == cfg["batch"]:  # the capture is of this workload only
            traffic = json.loads(tf.read_text()).get("mean_dram_bytes_per_launch")
        roofline = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (all launches of one step)", "achieved": ach,
                    "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic,
                    "traffic_source": "profiles/r02_gemm_traffic.json (mean dram read+write bytes per launch)" if traffic else None,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained",
                    "timed": "CUDA events around every b200_gemm launch of one eagerly launched step (same kernels as the graph "
                             "replay); raw event time: each pair also brackets the launch dispatch (~4 us per launch), nothing subtracted",
                    "gemm_launches": len(prof), "gemm_ms_per_step": gemm_ms, "gemm_tflop_per_step": flops / 1e12}
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        rooflines_hbm = []
        groups = {}
        for name, nbytes, a, b in kprof:
            g = groups.setdefault(name, [0, 0.0, 0.0])
            g[0] += 1; g[1] += nbytes; g[2] += a.elapsed_time(b)
        loss_b = sum(groups[n][1] for n in ("row_lse", "dino_ce") if n in groups)
        loss_ms = sum(groups[n][2] for n in ("row_lse", "dino_ce") if n in groups)
        if loss_ms > 0:
            rooflines_hbm.append({"bound": "hbm", "kernel": "dino_ce+row_lse (loss path of one step)", "achieved": loss_b / (loss_ms * 1e-3) / 1e9,
                                  "peak": hbm_peak, "unit": "GB/s", "frac": loss_b / (loss_ms * 1e-3) / 1e9 / hbm_peak,
                                  "algorithmic_bytes": loss_b, "ms": loss_ms, "launches": sum(groups[n][0] for n in ("row_lse", "dino_ce") if n in groups),
                                  "bytes_model": "2*K per teacher row (row_lse) + 2*K read + 2*K gradient write per student row (dino_ce); "
                                                 "teacher re-reads by dino_ce are L2 hits by design and not counted (SURVEY 8d)"})
        for n, label, model in (("adamw_ema", "adamw_ema (clip + AdamW + EMA + bf16 shadows, one sweep)",
                                 "20 B read (p,g,m,v,teacher) + 16 B fp32 write + 4 B bf16 write per parameter"),
                                ("sumsq", "sumsq (gradient norm)", "4 B read per parameter")):
            if n in groups and groups[n][2] > 0:
                g = groups[n]
                rooflines_hbm.append({"bound": "hbm", "kernel": label, "achieved": g[1] / (g[2] * 1e-3) / 1e9, "peak": hbm_peak,
                                      "unit": "GB/s", "frac": g[1] / (g[2] * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes": g[1],
                                      "ms": g[2], "launches": g[0], "bytes_model": model})
        for r in rooflines_hbm:
            r["peak_source"] = "MEASURED_PEAKS.json hbm_gbs (copy bandwidth)" if peaks else "fallback 6.65 TB/s"

    parity = None
    if rank == 0 and world == 1 and not args.no_parity:
        try:
            parity = bench_parity(method, cfg, batches[0]["views"], dev)
        except Exception as e:  # a checker problem must not take the measured line down
            parity = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()

    cpu_baseline = None
    gpu_torch_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:  # reported at N=1 only (the other ranks would idle)
        try:
            v, desc = cpu_reference(cfg, 1, 1, sweep=False)
            cpu_baseline = {"value": v, "unit": "images/s", **desc}
        except Exception as e:
            cpu_baseline = {"error": repr(e)[:300]}
    if rank == 0 and world == 1 and not args.no_gpu_baseline:
        from oracle import ref_full
        if ref_full.available():
            try:
                sec = reference_step_time(cfg, B, 5, 3, 0, device=str(dev))
                gpu_torch_baseline = {"value": B / sec, "unit": "images/s", "ms_per_step": sec * 1e3, "mode": "eager",
                                      "what": "the reference's own DINOv2 method class (same modules as cpu_baseline) on this B200 under "
                                              "torch.autocast(bf16), full step incl. its AdamW / clipping / EMA hooks, bs=%d, inputs resident, "
                                              "3 warm-up + 5 timed steps, CUDA events" % B}
            except Exception as e:  # the baseline must never take the bench line down
                gpu_torch_baseline = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()

    if rank == 0:
        line = {
            "metric": cfg["metric"], "value": value, "unit": "images/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": cfg["workload"] % B,
                       "global_batch": B * world, "parallelism": f"dp{world}",
                       "l2_policy": "inputs (2 alternating batches, 134 MB each at cfg2) and activations (>8 GB/step) exceed the 126 MB L2"},
            "clocks": clk.summary(), "e2e": e2e, "gpu_launches": launches,
            "gpu_launches_scope": "library kernel launches of rank 0 (graph replays counted per captured launch)",
            "host_ms_per_step": round(host_ms, 3), "loss": loss_val, "parity": parity,
            "roofline": roofline, "rooflines_hbm": rooflines_hbm, "cpu_baseline": cpu_baseline, "gpu_torch_baseline": gpu_torch_baseline,
        }
        if os.environ.get("B200_BENCH_DIAG_NO_ALLREDUCE", "0") == "1":
            line["diagnostic"] = "gradient all-reduce DISABLED (B200_BENCH_DIAG_NO_ALLREDUCE=1): not a training step, not a bench value"
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.cuda.synchronize()
        method.release_graphs()  # captured NCCL kernels (B200_GRAPH_NCCL=1) must be gone before the communicator is
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
