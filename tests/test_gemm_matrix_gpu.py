"""b200_gemm, instantiation by instantiation, against an exact fp64 reference.

Every case runs one (schedule, tile width, epilogue) kernel of csrc/gemm_tcgen05.cu on operands that are windows into
larger buffers: the input padding is bf16 NaN (a read past M, N or K poisons the result) and the outputs sit inside a
guard band of finite sentinels that must come back bitwise unchanged.

Reference: C64 = A @ B^T in fp64 on the device (bf16 products are exact in fp64) and S = |A| @ |B|^T, which scales
the accumulation bound: an fp32 result must satisfy |C - C64| <= TAU * |alpha| * S per element.  bf16 results may be
1 bf16 ulp from the fp64 value on top of that.  Staged epilogues are checked stage by stage against the kernel's own
earlier stage (u = bf16(acc + bias) is the second output), so one ulp of slack does not compound.

The tests without the gpu marker are pure torch and also run on a CPU: one asserts that the instantiation matrix
covers every kernel the dispatcher can launch, the others feed the comparison helper deliberately wrong outputs and
assert that it rejects each of them.
"""
from __future__ import annotations

import math
import re
import sys
import time
from dataclasses import dataclass, replace
from pathlib import Path

import pytest
import torch

from lightly_train_b200 import _lib

HAS_CUDA = torch.cuda.is_available()
gpu = pytest.mark.gpu
needs_cuda = pytest.mark.skipif(not HAS_CUDA, reason="needs CUDA")

EPI = {"bf16": _lib.EPI_BF16, "f32": _lib.EPI_F32, "f32_atomic": _lib.EPI_F32_ATOMIC, "bias_gelu": _lib.EPI_BIAS_GELU,
       "residual": _lib.EPI_RESIDUAL, "dgelu": _lib.EPI_DGELU, "bias_gelu_dg": _lib.EPI_BIAS_GELU_DG,
       "mul_aux": _lib.EPI_MUL_AUX}
SCHED = {"generic": 2, "ws": 1, "pair": 3}  # ws_mode that forces each schedule; 0 = the dispatcher chooses
WIDTHS = (128, 192, 256)
BLOCK_M, BLOCK_K = 128, 64
WS_MAX_K = {128: 384, 192: 384, 256: 256}  # the weight-stationary B slab must fit in shared memory

# Accumulation bound relative to S = |A| @ |B|^T.  Largest err / S of an fp32 output measured over this module on a
# B200 (1000 W power limit): generic 1.8e-7, weight-stationary 2.0e-7, CTA-pair 3.1e-7, dispatcher-chosen kernels
# 3.9e-7 (split-K atomics, K up to 65536).  TAU = 3.8e-6 leaves ~10x headroom; a dropped 64-wide k-block at
# K = 25216 gives ~5e-4 * S (asserted below to stay >= 20 * TAU).
TAU = 2.0 ** -18
F32_EPS = 2.0 ** -24
# The GELU epilogues use Abramowitz-Stegun 7.1.28 for erfc (csrc/common.cuh: gelu_tail).  Over every bf16 input
# u >= -4 the bf16 gelu(u) and gelu'(u) are within 1 bf16 ulp of the exact value.  Below -4 the approximation's
# relative error grows (gelu(-5): 10 ulps, gelu(-6): 63 ulps) while staying tiny in absolute terms: over all bf16
# u in [-8, -4] the error beyond 1 ulp is at most 2.2e-7 for gelu and 6e-10 for gelu'.  These allowances cover that
# tail; the test inputs keep |u| well below 8.  Measured on the B200 over this module: gelu up to 17.7 ulps (in the
# u < -4 tail), gelu' and dgelu 0.5 ulps.
GELU_EXCESS = 3e-7
GELU_GRAD_EXCESS = 1e-7
GELU_GRAD_F32 = 3e-7  # |gelu'_kernel(u) - gelu'(u)| before its bf16 rounding (DGELU multiplies the fp32 value)

# largest observed err / S per schedule (fp32 outputs) and largest gelu-stage error in bf16 ulps per epilogue
STATS: dict[str, float] = {}
BITWISE_ACROSS_SCHEDULES: dict[str, bool] = {}


# ----------------------------------------------------------------------------------------------- reference helpers
def bf16_round(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.bfloat16).double()


def bf16_ulp(x: torch.Tensor) -> torch.Tensor:
    """Spacing of bf16 numbers at |x| (8 significant bits); subnormal range clamped."""
    _, e = torch.frexp(x.double())
    u = torch.ldexp(torch.ones_like(x, dtype=torch.float64), (e - 8).clamp_min(-133))
    return torch.where(x == 0, torch.full_like(u, 2.0 ** -133), u)


def gelu64(u: torch.Tensor) -> torch.Tensor:
    return 0.5 * u * torch.special.erfc(-u / math.sqrt(2.0))


def gelu_grad64(u: torch.Tensor) -> torch.Tensor:
    return 0.5 * torch.special.erfc(-u / math.sqrt(2.0)) + u * torch.exp(-0.5 * u * u) / math.sqrt(2.0 * math.pi)


def fp64_products(A: torch.Tensor, B: torch.Tensor, budget: int = 1 << 23):
    """Yield (r0, r1, A[r0:r1] @ B^T, |A[r0:r1]| @ |B|^T) in fp64, a few row chunks at a time (<= ~1 GB of fp64)."""
    M, K = A.shape
    N = B.shape[0]
    B64 = B.double()
    B64a = B64.abs()
    rows = max(1, min(M, budget // max(N, K)))
    for r0 in range(0, M, rows):
        r1 = min(M, r0 + rows)
        a = A[r0:r1].double()
        yield r0, r1, a @ B64.t(), a.abs() @ B64a.t()


class Mismatch:
    """Collects element checks |got - want| <= tol; NaN anywhere counts as a failure."""

    def __init__(self, what: str):
        self.what, self.bad, self.total, self.worst = what, 0, 0, None

    def add(self, name: str, r0: int, got: torch.Tensor, want: torch.Tensor, tol: torch.Tensor) -> torch.Tensor:
        err = (got - want).abs()
        bad = ~(err <= tol)
        n = int(bad.sum())
        self.total += got.numel()
        if n:
            self.bad += n
            score = torch.where(bad, torch.nan_to_num(err / tol, nan=math.inf), torch.zeros_like(err))
            i = int(score.argmax())
            r, c = divmod(i, got.shape[1])
            self.worst = (f"{name}[{r0 + r}, {c}] = {float(got.flatten()[i])!r}, want {float(want.flatten()[i])!r} "
                          f"+- {float(tol.flatten()[i]):.3e} ({n} bad)")
        return err

    def raise_if_bad(self) -> None:
        assert self.bad == 0, f"{self.what}: {self.bad} / {self.total} elements outside tolerance; worst {self.worst}"


def _note(key: str, value: float) -> None:
    if value == value:
        STATS[key] = max(STATS.get(key, 0.0), value)


def check_gemm(epi: str, A: torch.Tensor, B: torch.Tensor, *, C: torch.Tensor, C2: torch.Tensor | None = None,
               aux: torch.Tensor | None = None, bias: torch.Tensor | None = None, gamma: torch.Tensor | None = None,
               rowscale: torch.Tensor | None = None, rows_per_scale: int = 1, alpha: float = 1.0,
               C0: torch.Tensor | None = None, n_add: int = 1, stage: torch.Tensor | None = None,
               label: str = "") -> None:
    """Check a b200_gemm result C (and C2) against epilogue(alpha * A @ B^T) in fp64.

    A [M, K] and B [N, K] are the logical bf16 operands (views of the stored ones).  C0: what an F32_ATOMIC output
    held before the call; n_add: an upper bound on the split-K partial sums added into it.  The residual and GELU
    epilogues need C2 (their stage u); without C2 the caller compares with a run that had it.  DGELU, MUL_AUX and
    BIAS_GELU_DG do not write their bf16 stage r = bf16(alpha * acc + bias): `stage` is r as the same kernel family
    writes it with the BF16 / BIAS_GELU epilogue, and without it the bound widens by the stage's rounding."""
    M, N = C.shape
    m = Mismatch(f"{label} {epi}")
    m2 = Mismatch(f"{label} {epi} (second output)")
    ms = Mismatch(f"{label} {epi} (bf16 stage)")
    bias64 = bias.double() if bias is not None else None
    for r0, r1, acc, S in fp64_products(A, B):
        x = alpha * acc
        if bias64 is not None:
            x = x + bias64
        aS = abs(alpha) * S
        dacc = TAU * aS
        c = C[r0:r1].double()
        if epi == "f32":
            err = m.add("C", r0, c, x, dacc + F32_EPS * x.abs())
            _note(f"err/S {label.split(':')[0]}", float(((err - F32_EPS * x.abs()).clamp_min(0) / aS).max()))
        elif epi == "f32_atomic":
            c0 = C0[r0:r1].double()
            err = m.add("C", r0, c, c0 + x, dacc + n_add * F32_EPS * (c0.abs() + aS))
            _note(f"err/S {label.split(':')[0]}",
                  float(((err - n_add * F32_EPS * (c0.abs() + aS)).clamp_min(0) / aS).max()))
        elif epi == "bf16":
            m.add("C", r0, c, x, bf16_ulp(x) + dacc)
        elif epi in ("bias_gelu", "residual"):
            assert C2 is not None, "the staged check reads the first stage from C2"
            u = C2[r0:r1].double()
            m2.add("C2", r0, u, x, bf16_ulp(x) + dacc)
            if epi == "bias_gelu":
                g = gelu64(u)
                err = m.add("C", r0, c, g, bf16_ulp(g) + GELU_EXCESS)
                _note("ulps gelu", float((err / bf16_ulp(g)).max()))
            else:
                rs = torch.ones(r1 - r0, 1, dtype=torch.float64, device=c.device)
                if rowscale is not None:
                    rs = rowscale.double()[torch.arange(r0, r1, device=c.device) // rows_per_scale][:, None]
                o = u * (gamma.double() if gamma is not None else 1.0) * rs
                a64 = aux[r0:r1].double()
                m.add("C", r0, c, a64 + o, 2.0 ** -22 * (a64.abs() + o.abs()))
        elif epi in ("dgelu", "mul_aux", "bias_gelu_dg"):
            a64 = aux[r0:r1].double() if aux is not None else None
            if stage is not None:
                # the kernel's own bf16 stage r = bf16(alpha * acc + bias), from the same kernel family
                r = stage[r0:r1].double()
                ms.add("stage", r0, r, x, bf16_ulp(x) + dacc)
                if epi == "bias_gelu_dg":
                    g = gelu64(r)
                    err = m.add("C", r0, c, g, bf16_ulp(g) + GELU_EXCESS)
                    _note("ulps gelu", float((err / bf16_ulp(g)).max()))
                    if C2 is not None:
                        gp = gelu_grad64(r)
                        err = m2.add("C2", r0, C2[r0:r1].double(), gp, bf16_ulp(gp) + GELU_GRAD_EXCESS)
                        _note("ulps gelu'", float((err / bf16_ulp(gp)).max()))
                else:
                    g, eps = (gelu_grad64(a64), GELU_GRAD_F32) if epi == "dgelu" else (a64, 0.0)
                    y = r * g
                    err = m.add("C", r0, c, y, bf16_ulp(y) + r.abs() * eps)
                    if epi == "dgelu":
                        _note("ulps dgelu", float(((err - r.abs() * eps).clamp_min(0) / bf16_ulp(y)).max()))
            else:
                # no stage to read: the kernel's bf16 rounding of x lies within w of x, so allow the function's
                # largest slope times w (|gelu'| <= 1.13, |gelu''| <= 0.8, d(r * g)/dr = g)
                w = dacc + bf16_ulp(x)
                if epi == "bias_gelu_dg":
                    g = gelu64(x)
                    m.add("C", r0, c, g, bf16_ulp(g) + GELU_EXCESS + 1.13 * w)
                    if C2 is not None:
                        gp = gelu_grad64(x)
                        m2.add("C2", r0, C2[r0:r1].double(), gp, bf16_ulp(gp) + GELU_GRAD_EXCESS + 0.8 * w)
                else:
                    g, eps = (gelu_grad64(a64), GELU_GRAD_F32) if epi == "dgelu" else (a64, 0.0)
                    y = x * g
                    m.add("C", r0, c, y, bf16_ulp(y) + g.abs() * w + (x.abs() + w) * eps)
        else:
            raise ValueError(epi)
    ms.raise_if_bad()
    m.raise_if_bad()
    m2.raise_if_bad()


# ----------------------------------------------------------------------------------------------- guarded buffers
class Guarded:
    """A [rows, cols] window into a larger buffer: `pre` whole rows before, `post` after, a leading column offset of
    `col_off` (a multiple of 8: keeps 16-byte alignment) and a row pitch of at least cols + 8 (a multiple of 8)."""

    def __init__(self, rows: int, cols: int, dtype: torch.dtype, device, fill: float, pre: int = 2, post: int = 1,
                 col_off: int = 8, extra_cols: int = 16):
        pitch = (cols + 7) // 8 * 8 + col_off + extra_cols
        self.buf = torch.full((pre + rows + post, pitch), fill, dtype=dtype, device=device)
        self.sl = (slice(pre, pre + rows), slice(col_off, col_off + cols))
        self.win = self.buf[self.sl]

    def snapshot(self) -> None:
        self.before = self.buf.clone()

    def assert_guard_intact(self, what: str, window_too: bool = False) -> None:
        want = self.before.clone()
        if not window_too:
            want[self.sl] = self.buf[self.sl]
        ity = {2: torch.int16, 4: torch.int32}[self.buf.element_size()]
        same = want.view(ity) == self.buf.view(ity)
        if not bool(same.all()):
            r, c = divmod(int((~same).flatten().nonzero()[0]), self.buf.shape[1])
            raise AssertionError(f"{what}: {int((~same).sum())} elements changed outside the window "
                                 f"(first at buffer [{r}, {c}]: {float(self.buf[r, c])!r})")


def poisoned(rows: int, cols: int, values: torch.Tensor, device) -> torch.Tensor:
    """bf16 [rows, cols] operand as a window into a NaN-padded buffer: lda = cols + 64 (rounded up to 8), padding
    rows before and after, a leading column offset of 8."""
    g = Guarded(rows, cols, torch.bfloat16, device, float("nan"), pre=1, post=2, col_off=8, extra_cols=56)
    g.win.copy_(values)
    return g.win


# ----------------------------------------------------------------------------------------------- cases
@dataclass(frozen=True)
class Case:
    name: str
    M: int
    N: int
    K: int
    epi: str
    sched: str = "auto"      # generic | ws | pair | auto
    bn: int = 0
    a_mn: int = 0
    b_mn: int = 0
    splits: int = 1
    alpha: float = 1.0
    bias: bool = False
    out2: bool = False
    gamma: bool = False
    rowscale: bool = False
    rows_per_scale: int = 1
    seed: int = 0


OPTIONAL = {"bf16": ("bias",), "f32": ("bias",), "f32_atomic": (), "bias_gelu": ("bias", "out2"),
            "residual": ("bias", "out2", "gamma", "rowscale"), "dgelu": (), "bias_gelu_dg": ("bias", "out2"),
            "mul_aux": ()}
# three option sets per (schedule, epilogue), one per tile width: every optional input is on in one and off in another
VARIANTS = ({"bias": True, "out2": True, "gamma": True, "rowscale": True, "alpha": 1.0},
            {"bias": False, "out2": False, "gamma": False, "rowscale": False, "alpha": 0.5},
            {"bias": False, "out2": True, "gamma": False, "rowscale": True, "alpha": 1.0})


def _matrix_a() -> list[Case]:
    """Every (schedule, tile width, epilogue) instantiation, at a shape with M, N and K tails."""
    out = []
    for s in SCHED:
        for i, w in enumerate(WIDTHS):
            for e in EPI:
                v = VARIANTS[i]
                opts = {k: v[k] for k in OPTIONAL[e]}
                pair_mn_ok = not (s == "pair" and w % 128)
                a_mn = b_mn = 0
                splits = 1
                if e in ("dgelu", "mul_aux") and pair_mn_ok:
                    b_mn = 1                     # the data-gradient layout
                if e == "f32_atomic":
                    a_mn, b_mn = 1, int(pair_mn_ok)  # the weight-gradient layout
                    splits = 2 if (i == 1 and s != "ws") else 1
                out.append(Case(f"{s}-{w}-{e}", M=300, N=w + 72, K=200, epi=e, sched=s, bn=w, a_mn=a_mn, b_mn=b_mn,
                                splits=splits, alpha=v["alpha"], rows_per_scale=37, seed=len(out), **opts))
    return out


def _matrix_b() -> list[Case]:
    """Operand layouts, M / N / K tails, the smallest shapes and long persistent loops, for each schedule."""
    out = []

    def add(name, **kw):
        out.append(Case(name, seed=1000 + len(out), **kw))

    for s, w in (("generic", 192), ("ws", 128), ("pair", 256)):
        kmax = WS_MAX_K[w] if s == "ws" else 10 ** 9
        for am in (0, 1):
            for bm in (0, 1):
                add(f"{s}-layout-a{am}b{bm}", M=333, N=2 * w + 8, K=200, epi="f32", sched=s, bn=w, a_mn=am, b_mn=bm,
                    bias=True)
        for t in (1, 31, 32, 33, 127):
            resid = t in (1, 33)
            add(f"{s}-mtail{t}", M=256 + t, N=w + w // 2 + 8, K=72, epi="residual" if resid else "bf16", sched=s,
                bn=w, bias=True, out2=resid, gamma=resid, rowscale=resid, rows_per_scale=37)
        if s == "pair":
            for t, what in ((100, "second-half-empty"), (128, "leader-exact"), (200, "in-second-half")):
                add(f"pair-tail-{what}", M=512 + t, N=w + 8, K=136, epi="f32", sched=s, bn=w, a_mn=1, b_mn=1)
        for r in (8, w // 2 + 8):
            add(f"{s}-ntail{r}", M=260, N=2 * w + r, K=136, epi="f32", sched=s, bn=w, bias=True)
        for k in (8, 40, 72, 200, 520):
            if k <= kmax:
                add(f"{s}-ktail{k}", M=260, N=w + 8, K=k, epi="bf16", sched=s, bn=w, a_mn=int(k == 40),
                    b_mn=int(k == 72))
        for am in (0, 1):
            add(f"{s}-smallest-a{am}b{am}", M=1, N=8, K=8 + 32 * am, epi="f32", sched=s, bn=w, a_mn=am, b_mn=am)
        # >= 3 tiles per CTA: the accumulator double buffer wraps several times and the ws kernel reloads B slabs
        add(f"{s}-many-tiles", M=3840, N=2048, K=256, epi="bf16", sched=s, bn=128, bias=True)
    for w in (256, 128, 192):
        add(f"ws-maxk-{w}", M=1000, N=w * 3 + 8, K=WS_MAX_K[w], epi="f32", sched="ws", bn=w)
    # the CTA-pair kernel at the shapes, operand majors and epilogue sequence it was first brought up with
    for (M, N, K, am, bm, w) in ((1000, 1152, 384, 0, 0, 192), (1100, 392, 72, 0, 0, 128), (384, 1152, 1000, 1, 1, 256),
                                 (512, 256, 128, 1, 0, 128)):
        add(f"pair-bringup-{M}x{N}x{K}-a{am}b{bm}", M=M, N=N, K=K, epi="f32", sched="pair", bn=w, a_mn=am, b_mn=bm)
        if not am and not bm:
            add(f"pair-bringup-{M}x{N}x{K}-splitk3", M=M, N=N, K=K, epi="f32_atomic", sched="pair", bn=w, splits=3)
            add(f"pair-bringup-{M}x{N}x{K}-residual", M=M, N=N, K=K, epi="residual", sched="pair", bn=w, bias=True,
                out2=True, gamma=True)
    return out


def _matrix_splitk() -> list[Case]:
    """F32_ATOMIC split-K: K = 1000 has 16 k-blocks; 3 and 5 do not divide it, 16 is every block, 40 is clamped."""
    out = []
    for s, w in (("generic", 192), ("pair", 128)):
        for sp in (3, 5, 16, 40):
            mn = int(sp in (5, 40))
            out.append(Case(f"{s}-splits{sp}", M=300, N=392, K=1000, epi="f32_atomic", sched=s, bn=w, a_mn=mn,
                            b_mn=mn, splits=sp, alpha=0.5 if sp == 3 else 1.0, seed=2000 + len(out)))
    return out


def _matrix_auto() -> list[Case]:
    """The product's GEMMs through the dispatcher's own choices (ws_mode = 0, block_n = 0, the product's splits).

    cfg2 (ViT-S/16, D 384, MLP 1536, 2 x 224^2 + 8 x 96^2 crops, batch 64): 25216 global tokens (197 per image),
    18944 local tokens (37 per image), 25088 / 18432 patch rows (K = 3 * 16 * 16); projection head 2048 / 256 / 65536
    on ~1000 rows.  See _models/dinov2_vit.py (forward :255-330, backward :394-413, wgrad :546-553, patch embed
    :448, :669-672) and _methods/dinov2/dinov2_head.py (:91-139)."""
    T, Tl, D, H = 25216, 18944, 384, 1536
    R, Hh, Bn, Ko = 1000, 2048, 256, 65536
    cs = [
        # forward
        ("cfg2-qkv", dict(M=T, N=3 * D, K=D, epi="bf16", bias=True)),
        ("cfg2-proj", dict(M=T, N=D, K=D, epi="residual", bias=True, out2=True, gamma=True, rowscale=True,
                           rows_per_scale=197)),
        ("cfg2-fc1", dict(M=T, N=H, K=D, epi="bias_gelu_dg", bias=True, out2=True)),
        ("cfg2-fc2", dict(M=T, N=D, K=H, epi="residual", bias=True, out2=True, gamma=True, rowscale=True,
                          rows_per_scale=197)),
        ("cfg2-fc2-teacher", dict(M=T, N=D, K=H, epi="residual", bias=True, gamma=True)),
        ("cfg2-local-proj", dict(M=Tl, N=D, K=D, epi="residual", bias=True, out2=True, gamma=True, rowscale=True,
                                 rows_per_scale=37)),
        ("cfg2-patch-embed", dict(M=25088, N=D, K=768, epi="bf16", bias=True)),
        # backward data gradients (weights read MN-major)
        ("cfg2-dfc2", dict(M=T, N=H, K=D, epi="mul_aux", b_mn=1)),
        ("cfg2-dfc1", dict(M=T, N=D, K=H, epi="bf16", b_mn=1)),
        ("cfg2-dproj", dict(M=T, N=D, K=D, epi="bf16", b_mn=1)),
        ("cfg2-dqkv", dict(M=T, N=D, K=3 * D, epi="bf16", b_mn=1)),
        # weight gradients: dW[out, in] += dy^T x, both operands MN-major, automatic split-K
        ("cfg2-wgrad-qkv", dict(M=3 * D, N=D, K=T, epi="f32_atomic", a_mn=1, b_mn=1, splits=0)),
        ("cfg2-wgrad-proj", dict(M=D, N=D, K=T, epi="f32_atomic", a_mn=1, b_mn=1, splits=0)),
        ("cfg2-wgrad-fc1", dict(M=H, N=D, K=T, epi="f32_atomic", a_mn=1, b_mn=1, splits=0)),
        ("cfg2-wgrad-fc2", dict(M=D, N=H, K=T, epi="f32_atomic", a_mn=1, b_mn=1, splits=0)),
        ("cfg2-wgrad-local-qkv", dict(M=3 * D, N=D, K=Tl, epi="f32_atomic", a_mn=1, b_mn=1, splits=0)),
        ("cfg2-wgrad-patch", dict(M=D, N=768, K=25088, epi="f32_atomic", a_mn=1, b_mn=1, splits=0)),
        ("cfg2-wgrad-local-patch", dict(M=D, N=768, K=18432, epi="f32_atomic", a_mn=1, b_mn=1, splits=0)),
        # projection head
        ("head-mlp0", dict(M=R, N=Hh, K=D, epi="bias_gelu_dg", bias=True, out2=True)),
        ("head-mlp2", dict(M=R, N=Hh, K=Hh, epi="bias_gelu_dg", bias=True, out2=True)),
        ("head-mlp4", dict(M=R, N=Bn, K=Hh, epi="bf16", bias=True)),
        ("head-last", dict(M=R, N=Ko, K=Bn, epi="bf16")),  # 8 M-tiles, K = 256: the weight-stationary kernel
        ("head-dW-last", dict(M=Ko, N=Bn, K=R, epi="f32", a_mn=1, b_mn=1)),
        ("head-dzn", dict(M=R, N=Bn, K=Ko, epi="f32_atomic", b_mn=1, splits=8)),
        ("head-wgrad-mlp4", dict(M=Bn, N=Hh, K=R, epi="f32_atomic", a_mn=1, b_mn=1, splits=0)),
        ("head-wgrad-mlp2", dict(M=Hh, N=Hh, K=R, epi="f32_atomic", a_mn=1, b_mn=1, splits=0)),
        ("head-wgrad-mlp0", dict(M=Hh, N=D, K=R, epi="f32_atomic", a_mn=1, b_mn=1, splits=0)),
        ("head-dU1", dict(M=R, N=Hh, K=Bn, epi="mul_aux", b_mn=1)),
        ("head-dU0", dict(M=R, N=Hh, K=Hh, epi="mul_aux", b_mn=1)),
        ("head-dx", dict(M=R, N=D, K=Hh, epi="bf16", b_mn=1)),
        # cfg3 (ViT-B/14 reg4, SwiGLU hidden 2048, 261 tokens per global crop, batch 32) and cfg5 (ViT-L/16, batch 16)
        ("cfg3-qkv", dict(M=16704, N=3 * 768, K=768, epi="bf16", bias=True)),
        ("cfg3-w3", dict(M=16704, N=768, K=2048, epi="residual", bias=True, out2=True, gamma=True, rowscale=True,
                         rows_per_scale=261)),
        ("cfg5-qkv", dict(M=6304, N=3 * 1024, K=1024, epi="bf16", bias=True)),
        ("cfg5-fc2", dict(M=6304, N=1024, K=4096, epi="residual", bias=True, out2=True, gamma=True, rowscale=True,
                          rows_per_scale=197)),
        # shapes of the earlier plain and auto-pair tests
        ("plain-256x384x128", dict(M=256, N=384, K=128, epi="f32")),
        ("plain-1000x1152x384", dict(M=1000, N=1152, K=384, epi="f32")),
        ("plain-384x1152x1000-a1b1", dict(M=384, N=1152, K=1000, epi="f32", a_mn=1, b_mn=1)),
        ("plain-300x256x520-b1", dict(M=300, N=256, K=520, epi="f32", b_mn=1)),
        ("plain-136x392x72-a1", dict(M=136, N=392, K=72, epi="f32", a_mn=1)),
        ("auto-pair-18944x1152x384", dict(M=18944, N=1152, K=384, epi="f32")),
    ]
    return [Case(n, seed=3000 + i, **kw) for i, (n, kw) in enumerate(cs)]


MATRIX_A, MATRIX_B, MATRIX_SPLITK, MATRIX_AUTO = _matrix_a(), _matrix_b(), _matrix_splitk(), _matrix_auto()


# ----------------------------------------------------------------------------------------------- running a case
def _ops():
    from lightly_train_b200 import ops
    return ops


def _randn(g: torch.Generator, *shape, scale: float = 1.0) -> torch.Tensor:
    return torch.randn(*shape, generator=g) * scale


def _n_add(c: Case) -> int:
    kbt = (c.K + BLOCK_K - 1) // BLOCK_K
    if c.splits == 0:
        return max(1, kbt // 4)  # the automatic chooser never splits finer than 4 k-blocks per split
    return max(1, min(c.splits, kbt))


class Launch:
    """Inputs of one case, generated from the case's seed; launch() runs the kernel into fresh guarded outputs."""

    def __init__(self, c: Case, dev="cuda"):
        self.c, self.dev = c, dev
        g = torch.Generator().manual_seed(c.seed)
        M, N, K = c.M, c.N, c.K
        av = _randn(g, M, K).bfloat16()
        bv = _randn(g, N, K, scale=K ** -0.5).bfloat16()  # unit-variance accumulators
        self.a = poisoned(K, M, av.t(), dev) if c.a_mn else poisoned(M, K, av, dev)
        self.b = poisoned(K, N, bv.t(), dev) if c.b_mn else poisoned(N, K, bv, dev)
        self.A = self.a.t() if c.a_mn else self.a
        self.B = self.b.t() if c.b_mn else self.b
        f = lambda t: t.float().to(dev)  # noqa: E731
        self.bias = f(_randn(g, N, scale=0.5)) if c.bias else None
        self.gamma = f(_randn(g, N)) if c.gamma else None
        nrs = (M + c.rows_per_scale - 1) // c.rows_per_scale
        self.rowscale = f(torch.rand(nrs, generator=g) * 2) if c.rowscale else None
        self.aux = None
        if c.epi == "residual":
            self.aux = Guarded(M, N, torch.float32, dev, float("nan"))
            self.aux.win.copy_(_randn(g, M, N))
        elif c.epi == "dgelu":
            self.aux = Guarded(M, N, torch.bfloat16, dev, float("nan"))
            self.aux.win.copy_(_randn(g, M, N))
        elif c.epi == "mul_aux":
            self.aux = Guarded(M, N, torch.bfloat16, dev, float("nan"))
            self.aux.win.copy_(torch.rand(M, N, generator=g) * 1.3 - 0.2)
        self.C0 = f(_randn(g, M, N)) if c.epi == "f32_atomic" else None
        if self.aux is not None:
            self.aux.snapshot()

    def launch(self, out2: bool | None = None, **over):
        c = replace(self.c, **over)
        out2 = c.out2 if out2 is None else out2
        f32_out = c.epi in ("f32", "f32_atomic", "residual")
        C = Guarded(c.M, c.N, torch.float32 if f32_out else torch.bfloat16, self.dev, -1234.5)
        if c.epi == "f32_atomic":
            C.win.copy_(self.C0)
        else:
            C.win.fill_(float("nan"))  # an element the kernel skips stays NaN
        C2 = None
        if out2 and c.epi in ("bias_gelu", "residual", "bias_gelu_dg"):
            C2 = Guarded(c.M, c.N, torch.bfloat16, self.dev, -1234.5)
            C2.win.fill_(float("nan"))
        C.snapshot()
        if C2 is not None:
            C2.snapshot()
        aux = self.aux.win if c.epi in ("residual", "dgelu", "mul_aux") else None
        _ops().gemm(self.a, self.b, C.win, a_mn=bool(c.a_mn), b_mn=bool(c.b_mn), epi=EPI[c.epi], bias=self.bias,
                    out2=C2.win if C2 is not None else None, aux=aux,
                    gamma=self.gamma, rowscale=self.rowscale, rows_per_scale=c.rows_per_scale, alpha=c.alpha,
                    splits=c.splits, block_n=c.bn, ws_mode=SCHED.get(c.sched, 0))
        torch.cuda.synchronize()
        C.assert_guard_intact(f"{c.name}: C")
        if C2 is not None:
            C2.assert_guard_intact(f"{c.name}: C2")
        if self.aux is not None:
            self.aux.assert_guard_intact(f"{c.name}: aux (an input)", window_too=True)
        return C.win, (C2.win if C2 is not None else None)

    def stage(self):
        """The bf16 stage r = bf16(alpha * acc + bias) that DGELU / MUL_AUX / BIAS_GELU_DG compute but do not write, as
        the same schedule and tile width write it with the BF16 (or BIAS_GELU) epilogue.  With the schedule left to
        the dispatcher the two epilogues may run on different kernels, so there is none."""
        c = self.c
        if c.epi not in ("dgelu", "mul_aux", "bias_gelu_dg") or c.sched == "auto":
            return None
        if c.epi == "bias_gelu_dg":
            return self.launch(out2=True, epi="bias_gelu")[1]
        return self.launch(epi="bf16")[0]

    def check(self, C, C2):
        c = self.c
        check_gemm(c.epi, self.A, self.B, C=C, C2=C2, aux=self.aux.win if self.aux is not None else None,
                   bias=self.bias, gamma=self.gamma, rowscale=self.rowscale, rows_per_scale=c.rows_per_scale,
                   alpha=c.alpha, C0=self.C0, n_add=_n_add(c), stage=self.stage(), label=f"{c.sched}: {c.name}")


def _bitwise_equal(x: torch.Tensor, y: torch.Tensor) -> bool:
    ity = {2: torch.int16, 4: torch.int32}[x.element_size()]
    return bool((x.contiguous().view(ity) == y.contiguous().view(ity)).all())


def run_case(c: Case) -> None:
    L = Launch(c)
    C, C2 = L.launch()
    staged = c.epi in ("bias_gelu", "residual", "bias_gelu_dg")
    if staged and C2 is None:
        # the branch without the second output: C must be bitwise what the same kernel writes with it
        Cw, C2w = L.launch(out2=True)
        L.check(Cw, C2w)
        assert _bitwise_equal(C, Cw), f"{c.name}: C differs between the launches with and without the second output"
    else:
        L.check(C, C2)
    if c.epi != "f32_atomic":
        Cr, C2r = L.launch()
        assert _bitwise_equal(C, Cr), f"{c.name}: a second launch on the same inputs changed C"
        if C2 is not None:
            assert _bitwise_equal(C2, C2r), f"{c.name}: a second launch on the same inputs changed C2"


@pytest.fixture(scope="module")
def _report():
    t0 = time.perf_counter()
    yield
    lines = [f"test_gemm_matrix_gpu: {time.perf_counter() - t0:.1f} s wall, "
             f"peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB"]
    lines += [f"  {k}: {v:.3e}" + (f"  (TAU = {TAU:.3e})" if k.startswith("err/S") else "") for k, v in sorted(STATS.items())]
    lines += [f"  bitwise equal across schedules, {k}: {v}" for k, v in sorted(BITWISE_ACROSS_SCHEDULES.items())]
    print("\n".join(lines), file=sys.stderr)


# ----------------------------------------------------------------------------------------------- GPU tests
@gpu
@needs_cuda
@pytest.mark.parametrize("case", MATRIX_A, ids=lambda c: c.name)
def test_instantiation(case, _report):
    run_case(case)


@gpu
@needs_cuda
@pytest.mark.parametrize("case", MATRIX_B, ids=lambda c: c.name)
def test_layout_and_tails(case, _report):
    run_case(case)


@gpu
@needs_cuda
@pytest.mark.parametrize("case", MATRIX_SPLITK, ids=lambda c: c.name)
def test_splitk(case, _report):
    run_case(case)


@gpu
@needs_cuda
def test_splitk_long_k_accumulates(_report):
    """A weight-gradient-like split-K GEMM at long K through the dispatcher's tile choice: 13 splits of 141 k-blocks
    (K = 9000 has a 40-wide tail), both operands MN-major, added into a pre-filled output."""
    run_case(Case("splitk13-1152x384x9000", M=1152, N=384, K=9000, epi="f32_atomic", a_mn=1, b_mn=1, splits=13,
                  seed=5000))


@gpu
@needs_cuda
@pytest.mark.parametrize("case", MATRIX_AUTO, ids=lambda c: c.name)
def test_auto_dispatch(case, _report):
    run_case(case)


@gpu
@needs_cuda
@pytest.mark.parametrize("epi", ["bf16", "f32"])
def test_schedules_agree(epi, _report):
    """The same inputs through the generic, weight-stationary and CTA-pair kernels: each passes the fp64 check and
    the three agree within the tolerance.  On a B200 they are in fact bitwise equal; the report records it, the test
    does not require it."""
    base = Case(f"agree-{epi}", M=1000, N=1024, K=256, epi=epi, bn=128, bias=True, seed=4000)
    L = Launch(base)
    outs = {}
    for s in SCHED:
        L.c = replace(base, sched=s)
        outs[s], _ = L.launch()
        L.check(outs[s], None)
    x = L.A.double() @ L.B.double().t() + L.bias.double()
    S = L.A.double().abs() @ L.B.double().abs().t()
    tol = 2 * TAU * S + 2 * F32_EPS * x.abs() if epi == "f32" else 2 * bf16_ulp(x) + 2 * TAU * S
    for s in ("ws", "pair"):
        d = (outs[s].double() - outs["generic"].double()).abs()
        assert bool((d <= tol).all()), f"{s} vs generic: {int((d > tol).sum())} elements differ beyond the tolerance"
        BITWISE_ACROSS_SCHEDULES[f"{epi} {s} vs generic"] = _bitwise_equal(outs[s], outs["generic"])


REFUSALS = [
    # (id, case, what b200_gemm returns)
    ("ws-k-above-384", Case("r", M=1000, N=256, K=448, epi="bf16", sched="ws", bn=128), "UNSUPPORTED"),
    ("ws-256-k-above-256", Case("r", M=1000, N=256, K=320, epi="bf16", sched="ws", bn=256), "UNSUPPORTED"),
    ("ws-splitk", Case("r", M=1000, N=256, K=256, epi="f32_atomic", sched="ws", bn=128, splits=2), "INVALID_ARG"),
    ("pair-bmn-192", Case("r", M=512, N=384, K=128, epi="f32", sched="pair", bn=192, b_mn=1), "UNSUPPORTED"),
    ("splitk-non-atomic", Case("r", M=256, N=256, K=512, epi="f32", splits=2), "INVALID_ARG"),
    ("residual-no-aux", Case("r", M=256, N=256, K=128, epi="residual"), "INVALID_ARG"),
    ("dgelu-no-aux", Case("r", M=256, N=256, K=128, epi="dgelu"), "INVALID_ARG"),
    ("mul-aux-no-aux", Case("r", M=256, N=256, K=128, epi="mul_aux"), "INVALID_ARG"),
    ("misaligned-a", Case("r", M=256, N=256, K=128, epi="f32"), "UNSUPPORTED"),
]


@gpu
@needs_cuda
@pytest.mark.parametrize("rid,case,code", REFUSALS, ids=[r[0] for r in REFUSALS])
def test_refusals(rid, case, code):
    """Refused arguments raise B200Error before any launch: the output window and its guard band stay untouched."""
    from lightly_train_b200._lib import B200Error
    ops = _ops()
    L = Launch(case)
    a = L.a
    if rid == "misaligned-a":  # a window that starts one element (2 bytes) past a 16-byte boundary
        base = poisoned(case.M, case.K + 8, torch.zeros(case.M, case.K + 8), "cuda")
        a = base[:, 1:1 + case.K]
    f32_out = case.epi in ("f32", "f32_atomic", "residual")
    C = Guarded(case.M, case.N, torch.float32 if f32_out else torch.bfloat16, "cuda", -1234.5)
    C.win.fill_(7.0)
    C.snapshot()
    with pytest.raises(B200Error, match=code):
        ops.gemm(a, L.b, C.win, a_mn=bool(case.a_mn), b_mn=bool(case.b_mn), epi=EPI[case.epi], bias=L.bias,
                 splits=case.splits, block_n=case.bn, ws_mode=SCHED.get(case.sched, 0))
    torch.cuda.synchronize()
    C.assert_guard_intact(rid, window_too=True)


# ----------------------------------------------------------------------------------------------- CPU tests
def _dispatchable_instantiations() -> set[tuple[str, int, str]]:
    """(schedule, tile width, epilogue) of every kernel b200_gemm can launch, read from csrc/gemm_tcgen05.cu."""
    src = (Path(__file__).resolve().parents[1] / "lightly_train_b200" / "csrc" / "gemm_tcgen05.cu").read_text()
    switch = re.search(r"#define B200_EPI_SWITCH\(CALL\)(.*?)default:", src, re.S).group(1)
    epi_names = {v: k for k, v in EPI.items()}
    epis = [epi_names[getattr(_lib, "EPI_" + n)] for n in re.findall(r"case B200_EPI_(\w+): return CALL", switch)]
    body = src[src.index('extern "C" int b200_gemm('):]
    sched_of = {"": "generic", "_ws": "ws", "_2sm": "pair"}
    kernels = {(sched_of[s], int(w)) for s, w in re.findall(r"return launch_gemm(_ws|_2sm)?<(\d+)", body)}
    return {(s, w, e) for s, w in kernels for e in epis}


def test_matrix_covers_every_instantiation():
    """One instantiation case per (schedule, tile width, epilogue) kernel the dispatcher can launch; adding a kernel
    to csrc/gemm_tcgen05.cu without a case here fails.  No instantiation is refused outright by the dispatcher (the
    CTA-pair kernel refuses only the MN-major B operand at width 192, a layout the matrix avoids there), so the
    exclusion list is empty."""
    excluded: set[tuple[str, int, str]] = set()
    want = _dispatchable_instantiations() - excluded
    assert len(want) == 3 * 3 * 8
    have = {(c.sched, c.bn, c.epi) for c in MATRIX_A}
    assert have == want, (sorted(want - have), sorted(have - want))
    assert len({c.name for c in MATRIX_A + MATRIX_B + MATRIX_SPLITK + MATRIX_AUTO}) == \
        len(MATRIX_A + MATRIX_B + MATRIX_SPLITK + MATRIX_AUTO)
    # every optional input of every epilogue is on in one case and off in another, per schedule
    for s in SCHED:
        for e, opts in OPTIONAL.items():
            cs = [c for c in MATRIX_A if c.sched == s and c.epi == e]
            for o in opts:
                assert {getattr(c, o) for c in cs} == {True, False}, (s, e, o)
        assert {c.alpha for c in MATRIX_A if c.sched == s} == {1.0, 0.5}
    # the forced cases stay inside what the dispatcher accepts (its refusals are test_refusals' business)
    assert all(c.K <= WS_MAX_K[c.bn] and c.splits == 1 for c in MATRIX_A + MATRIX_B if c.sched == "ws")
    assert not any(c.sched == "pair" and c.b_mn and c.bn == 192 for c in MATRIX_A + MATRIX_B + MATRIX_SPLITK)


def _cpu_operands(M, N, K, seed=0):
    g = torch.Generator().manual_seed(seed)
    A = _randn(g, M, K).bfloat16()
    B = _randn(g, N, K, scale=K ** -0.5).bfloat16()
    return A, B, A.double() @ B.double().t()


def test_negative_controls_are_rejected():
    """The comparison helper accepts the exact result and rejects each of these wrong "kernel outputs"."""
    A, B, x = _cpu_operands(300, 24, 25216)
    check_gemm("f32", A, B, C=x.float(), label="exact")
    # the product with its last k-block dropped: err / S must sit far above TAU
    dropped = A[:, :-BLOCK_K].double() @ B[:, :-BLOCK_K].double().t()
    S = A.double().abs() @ B.double().abs().t()
    assert float(((dropped - x).abs() / S).max()) >= 20 * TAU
    with pytest.raises(AssertionError):
        check_gemm("f32", A, B, C=dropped.float(), label="dropped k-block")
    # one row of the last M-tile zeroed
    bad = x.float().clone()
    bad[299] = 0
    with pytest.raises(AssertionError):
        check_gemm("f32", A, B, C=bad, label="zeroed row")
    # bias added twice
    bias = torch.randn(24, generator=torch.Generator().manual_seed(1)) * 0.5
    check_gemm("f32", A, B, C=(x + bias.double()).float(), bias=bias, label="bias once")
    with pytest.raises(AssertionError):
        check_gemm("f32", A, B, C=(x + 2 * bias.double()).float(), bias=bias, label="bias twice")
    # a NaN in a valid element
    bad = x.float().clone()
    bad[17, 5] = float("nan")
    with pytest.raises(AssertionError):
        check_gemm("f32", A, B, C=bad, label="NaN")


def test_negative_controls_bf16_and_guard():
    A, B, x = _cpu_operands(200, 64, 1000, seed=2)
    good = x.bfloat16()
    check_gemm("bf16", A, B, C=good, label="exact")
    # every element 2 bf16 ulps away from the correctly rounded value (in magnitude)
    off = (good.view(torch.int16) + 2).view(torch.bfloat16)
    with pytest.raises(AssertionError):
        check_gemm("bf16", A, B, C=off, label="2 ulps")
    # a single element 2 ulps off
    one = good.clone()
    one.view(torch.int16)[123 % 200, 7] += 2
    with pytest.raises(AssertionError):
        check_gemm("bf16", A, B, C=one, label="one element 2 ulps")
    # a staged epilogue: gelu of the kernel's own u, one element 2 ulps off
    u = x.bfloat16()
    h = gelu64(u.double()).bfloat16()
    check_gemm("bias_gelu", A, B, C=h, C2=u, label="gelu exact")
    h.view(torch.int16)[5, 9] += 2
    with pytest.raises(AssertionError):
        check_gemm("bias_gelu", A, B, C=h, C2=u, label="gelu 2 ulps")
    # a changed sentinel in the guard band
    g = Guarded(200, 64, torch.float32, "cpu", -1234.5)
    g.snapshot()
    g.win.copy_(x)
    g.assert_guard_intact("untouched")
    g.buf[1, 3] = -1234.0
    with pytest.raises(AssertionError):
        g.assert_guard_intact("sentinel changed")
