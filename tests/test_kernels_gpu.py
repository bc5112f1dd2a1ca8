"""Per-kernel numerics on the GPU: each C-ABI entry point against a plain PyTorch fp32 statement of the same
op (tolerances written per test; bf16 outputs are compared after rounding the reference the same way)."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs CUDA", allow_module_level=True)

from lightly_train_b200 import ops  # noqa: E402

dev = "cuda"


def rnd(*shape, scale=1.0, dtype=torch.float32, seed=None):
    g = torch.Generator(device="cpu")
    g.manual_seed(seed if seed is not None else hash(shape) % 10000)
    return (torch.randn(*shape, generator=g) * scale).to(dev).to(dtype)


def test_gemm_fused_epilogues():
    M, N, K = 777, 384, 1536
    a, b = rnd(M, K, dtype=torch.bfloat16, scale=0.5, seed=3), rnd(N, K, dtype=torch.bfloat16, scale=0.05, seed=4)
    bias, gamma, x = rnd(N, seed=5), rnd(N, seed=6), rnd(M, N, seed=7)
    rs = torch.rand(M // 37 + 1, device=dev)
    out, o2 = torch.empty(M, N, device=dev), torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    ops.gemm(a, b, out, epi=ops.EPI_RESIDUAL, bias=bias, out2=o2, aux=x, gamma=gamma, rowscale=rs, rows_per_scale=37)
    o = (a.float() @ b.float().t() + bias).bfloat16()
    torch.testing.assert_close(o2.float(), o.float(), rtol=2e-2, atol=2e-2)
    want = x + o2.float() * gamma * rs.repeat_interleave(37)[:M, None]
    torch.testing.assert_close(out, want, rtol=1e-5, atol=1e-5)
    # bias + gelu
    h, u = torch.empty(M, N, device=dev, dtype=torch.bfloat16), torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    ops.gemm(a, b, h, epi=ops.EPI_BIAS_GELU, bias=bias, out2=u)
    torch.testing.assert_close(h.float(), F.gelu(u.float()).bfloat16().float(), rtol=1e-2, atol=1e-2)
    # dgelu
    d = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    ops.gemm(a, b, d, epi=ops.EPI_DGELU, aux=u)
    uf = u.float().requires_grad_(True)
    F.gelu(uf).backward((a.float() @ b.float().t()).bfloat16().float())
    torch.testing.assert_close(d.float(), uf.grad, rtol=2e-2, atol=2e-2)


def test_gemm_saved_derivative_gelu_epilogues():
    """BIAS_GELU_DG stores gelu'(u) for the backward; MUL_AUX consumes it (same dU as the DGELU epilogue)."""
    M, N, K = 777, 1536, 384
    a, b = rnd(M, K, dtype=torch.bfloat16, scale=0.5, seed=3), rnd(N, K, dtype=torch.bfloat16, scale=0.05, seed=4)
    bias = rnd(N, seed=5)
    h, g = torch.empty(M, N, device=dev, dtype=torch.bfloat16), torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    ops.gemm(a, b, h, epi=ops.EPI_BIAS_GELU_DG, bias=bias, out2=g)
    u = (a.float() @ b.float().t() + bias).bfloat16().float().requires_grad_(True)
    hr = F.gelu(u)
    hr.sum().backward()
    torch.testing.assert_close(h.float(), hr.detach().bfloat16().float(), rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(g.float(), u.grad.bfloat16().float(), rtol=1e-2, atol=1e-2)
    dy = rnd(M, K, dtype=torch.bfloat16, seed=6)
    w = rnd(K, N, dtype=torch.bfloat16, scale=0.05, seed=7)  # [out=K... used as MN-major B: dU[M,N] = dy[M,K] @ w[K,N]
    dU = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    ops.gemm(dy, w, dU, b_mn=True, epi=ops.EPI_MUL_AUX, aux=g)
    want = (dy.float() @ w.float()).bfloat16().float() * g.float()
    torch.testing.assert_close(dU.float(), want.bfloat16().float(), rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("B,N,h", [(3, 197, 6), (5, 37, 2), (2, 261, 3), (2, 54, 2), (1, 16, 1)])
def test_attention_fwd_bwd(B, N, h):
    D = h * 64
    qkv = rnd(B * N, 3 * D, dtype=torch.bfloat16, scale=1.0, seed=10)
    out = torch.empty(B * N, D, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(B * h, N, device=dev)
    ops.attention_fwd(qkv, B, N, h, out, lse, 0.125)
    q5 = qkv.float().view(B, N, 3, h, 64).permute(2, 0, 3, 1, 4).clone().requires_grad_(True)
    q, k, v = q5[0] * 0.125, q5[1], q5[2]
    s = (q @ k.transpose(-1, -2))
    p = s.softmax(-1)
    o = (p @ v).transpose(1, 2).reshape(B * N, D)
    torch.testing.assert_close(out.float(), o, rtol=3e-2, atol=3e-2)
    torch.testing.assert_close(lse.view(B, h, N), torch.logsumexp(s, -1), rtol=1e-2, atol=3e-2)
    do = rnd(B * N, D, dtype=torch.bfloat16, scale=1.0, seed=11)
    o.backward(do.float())
    dqkv = torch.empty_like(qkv)
    ops.attention_bwd(qkv, out, do, lse, B, N, h, dqkv, 0.125)
    want = q5.grad.permute(1, 3, 0, 2, 4).reshape(B * N, 3 * D)
    err = (dqkv.float() - want).abs().max().item()
    assert err < 0.05 * max(1.0, want.abs().max().item()), err
    rel = (dqkv.float() - want).norm() / want.norm()
    assert rel < 2e-2, rel
    # fused qkv-bias gradient: += column sums of the (bf16) dqkv the kernel wrote, padded key rows excluded
    cs = torch.ones(3 * D, device=dev)
    dqkv2 = torch.empty_like(qkv)
    ops.attention_bwd(qkv, out, do, lse, B, N, h, dqkv2, 0.125, colsum=cs)
    assert torch.equal(dqkv2, dqkv)
    ref = dqkv.float().sum(0) + 1
    torch.testing.assert_close(cs, ref, rtol=1e-4, atol=1e-3 * max(1.0, float(ref.abs().max())))


@pytest.mark.parametrize("B,N,h", [(3, 197, 6), (2, 201, 3), (5, 37, 2), (2, 256, 3), (2, 130, 2), (1, 16, 1), (3, 128, 2), (4, 100, 1),
                                   (7, 54, 3), (40, 197, 16)])
def test_attention_fwd_tcgen05(B, N, h):
    """tcgen05 / TMEM / TMA forward (the product path for 128 < N <= 256) against the fp32 torch statement and against
    the warp-level kernel (P is rounded before normalisation here, so the two differ by bf16 rounding only)."""
    D = h * 64
    qkv = rnd(B * N, 3 * D, dtype=torch.bfloat16, scale=1.0, seed=10)
    out, ref = (torch.empty(B * N, D, device=dev, dtype=torch.bfloat16) for _ in range(2))
    lse, lse_ref = (torch.empty(B * h, N, device=dev) for _ in range(2))
    ops.attention_fwd_tc(qkv, B, N, h, out, lse, 0.125)
    saved = (ops.TC_ATTENTION_FWD, ops.TC_ATTENTION_PACKED)
    ops.TC_ATTENTION_FWD = ops.TC_ATTENTION_PACKED = False  # the warp-level (mma.sync) kernel for every length
    try:
        ops.attention_fwd(qkv, B, N, h, ref, lse_ref, 0.125)
    finally:
        ops.TC_ATTENTION_FWD, ops.TC_ATTENTION_PACKED = saved
    q5 = qkv.float().view(B, N, 3, h, 64).permute(2, 0, 3, 1, 4)
    s = (q5[0] * 0.125) @ q5[1].transpose(-1, -2)
    o = (s.softmax(-1) @ q5[2]).transpose(1, 2).reshape(B * N, D)
    torch.testing.assert_close(out.float(), o, rtol=3e-2, atol=3e-2)
    torch.testing.assert_close(lse.view(B, h, N), torch.logsumexp(s, -1), rtol=1e-2, atol=3e-2)
    torch.testing.assert_close(out.float(), ref.float(), rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(lse, lse_ref, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("B,N,h", [(3, 197, 6), (2, 201, 3), (5, 37, 2), (2, 208, 1), (2, 130, 2), (3, 128, 2), (4, 100, 1), (7, 54, 3),
                                   (1, 16, 1), (40, 197, 16)])
def test_attention_bwd_tcgen05(B, N, h):
    """tcgen05 backward (the product path for 128 < N <= 208): dq | dk | dv against torch autograd (fp32) and against the
    warp-level kernel, and the fused qkv-bias gradient against the column sums of the bf16 dqkv it wrote."""
    D = h * 64
    qkv = rnd(B * N, 3 * D, dtype=torch.bfloat16, scale=1.0, seed=10)
    do = rnd(B * N, D, dtype=torch.bfloat16, scale=1.0, seed=11)
    out = torch.empty(B * N, D, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(B * h, N, device=dev)
    ops.attention_fwd(qkv, B, N, h, out, lse, 0.125)
    q5 = qkv.float().view(B, N, 3, h, 64).permute(2, 0, 3, 1, 4).clone().requires_grad_(True)
    o = (((q5[0] * 0.125) @ q5[1].transpose(-1, -2)).softmax(-1) @ q5[2]).transpose(1, 2).reshape(B * N, D)
    o.backward(do.float())
    want = q5.grad.permute(1, 3, 0, 2, 4).reshape(B * N, 3 * D)
    dq_t, dq_w = torch.full_like(qkv, 7.0), torch.empty_like(qkv)
    cs = torch.ones(3 * D, device=dev)
    ops.attention_bwd_tc(qkv, out, do, lse, B, N, h, dq_t, 0.125, colsum=cs)
    saved = (ops.TC_ATTENTION_BWD, ops.TC_ATTENTION_PACKED)
    ops.TC_ATTENTION_BWD = ops.TC_ATTENTION_PACKED = False  # the warp-level (mma.sync) kernel for every length
    try:
        ops.attention_bwd(qkv, out, do, lse, B, N, h, dq_w, 0.125)
    finally:
        ops.TC_ATTENTION_BWD, ops.TC_ATTENTION_PACKED = saved
    assert torch.isfinite(dq_t.float()).all()
    for sl in (slice(0, D), slice(D, 2 * D), slice(2 * D, 3 * D)):
        a, w, t = dq_t[:, sl].float(), dq_w[:, sl].float(), want[:, sl]
        assert ((a - t).norm() / t.norm()).item() < 2e-2
        assert (a - t).abs().max().item() < 0.05 * max(1.0, t.abs().max().item())
        assert ((a - w).norm() / w.norm()).item() < 1e-2
    ref = dq_t.float().sum(0) + 1
    torch.testing.assert_close(cs, ref, rtol=1e-4, atol=1e-3 * max(1.0, float(ref.abs().max())))


@pytest.mark.parametrize("T,D", [(1000, 384), (77, 128), (300, 1024), (64, 192)])
def test_layernorm_fwd_bwd(T, D):
    x = rnd(T, D, seed=12, scale=2.0).requires_grad_(True)
    w, b = (1 + 0.1 * rnd(D, seed=13)).requires_grad_(True), rnd(D, seed=14).requires_grad_(True)
    y32, mean, rstd = torch.empty(T, D, device=dev), torch.empty(T, device=dev), torch.empty(T, device=dev)
    ops.layernorm_fwd(x.detach(), w.detach(), b.detach(), 1e-6, y32, mean, rstd)
    ref = F.layer_norm(x, (D,), w, b, 1e-6)
    torch.testing.assert_close(y32, ref, rtol=1e-5, atol=1e-5)
    y16 = torch.empty(T, D, device=dev, dtype=torch.bfloat16)
    ops.layernorm_fwd(x.detach(), w.detach(), b.detach(), 1e-6, y16)
    torch.testing.assert_close(y16.float(), ref.bfloat16().float(), rtol=1e-2, atol=1e-2)
    dy = rnd(T, D, seed=15)
    ref.backward(dy)
    dx = torch.ones(T, D, device=dev)
    dw, db = torch.zeros(D, device=dev), torch.zeros(D, device=dev)
    ops.layernorm_bwd(dy, x.detach(), w.detach(), mean, rstd, dx, True, dw, db)
    torch.testing.assert_close(dx, 1 + x.grad, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(dw, w.grad, rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(db, b.grad, rtol=1e-4, atol=1e-3)
    dx2 = torch.empty(T, D, device=dev)
    ops.layernorm_bwd(dy.bfloat16(), x.detach(), w.detach(), mean, rstd, dx2, False)
    torch.testing.assert_close(dx2, x.grad, rtol=5e-2, atol=5e-2)


def test_layernorm_bwd_fused_with_layerscale_bwd():
    T, D = 1003, 384
    x = rnd(T, D, seed=50, scale=2.0)
    w = 1 + 0.1 * rnd(D, seed=51)
    mean, rstd = torch.empty(T, device=dev), torch.empty(T, device=dev)
    y = torch.empty(T, D, device=dev)
    ops.layernorm_fwd(x, w, rnd(D, seed=52), 1e-6, y, mean, rstd)
    dy = rnd(T, D, dtype=torch.bfloat16, seed=53)
    o = rnd(T, D, dtype=torch.bfloat16, seed=54)
    gamma = rnd(D, seed=55)
    rs = torch.rand(T // 59 + 1, device=dev)
    dx0 = rnd(T, D, seed=56)
    # reference: the two separate kernels
    dx_ref = dx0.clone(); dw_r, db_r = torch.zeros(D, device=dev), torch.zeros(D, device=dev)
    ops.layernorm_bwd(dy, x, w, mean, rstd, dx_ref, True, dw_r, db_r)
    do_ref = torch.empty(T, D, device=dev, dtype=torch.bfloat16); dg_r, dbi_r = torch.zeros(D, device=dev), torch.zeros(D, device=dev)
    ops.layerscale_bwd(dx_ref, o, gamma, rs, 59, do_ref, dg_r, dbi_r)
    dx = dx0.clone(); dw, db = torch.zeros(D, device=dev), torch.zeros(D, device=dev)
    do = torch.empty(T, D, device=dev, dtype=torch.bfloat16); dg, dbi = torch.zeros(D, device=dev), torch.zeros(D, device=dev)
    ops.layernorm_bwd_ls(dy, x, w, mean, rstd, dx, True, dw, db, o, gamma, rs, 59, do, dg, dbi)
    torch.testing.assert_close(dx, dx_ref, rtol=1e-5, atol=1e-5)
    assert torch.equal(do, do_ref)
    for a, b in ((dw, dw_r), (db, db_r), (dg, dg_r), (dbi, dbi_r)):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("p,H", [(16, 224), (16, 96), (14, 98)])
def test_im2col(p, H):
    x = rnd(3, 3, H, H, seed=16)
    Np = (H // p) ** 2
    cols = torch.empty(3 * Np, 3 * p * p, device=dev, dtype=torch.bfloat16)
    ops.im2col(x, p, cols)
    want = F.unfold(x, kernel_size=p, stride=p).transpose(1, 2).reshape(3 * Np, 3 * p * p)
    assert torch.equal(cols, want.bfloat16())


@pytest.mark.parametrize("R", [0, 4])
def test_assemble_tokens_fwd_bwd(R):
    B, Np, D = 5, 36, 128
    N = 1 + R + Np
    tok = rnd(B * Np, D, dtype=torch.bfloat16, seed=17)
    masks = (torch.rand(B, Np, device=dev) < 0.3)
    mt, cls, pos = rnd(1, D, seed=18), rnd(D, seed=19), rnd(1 + Np, D, seed=20)
    reg = rnd(R, D, seed=21) if R else None
    x = torch.empty(B, N, D, device=dev)
    ops.assemble_tokens(tok, masks.to(torch.uint8), mt, cls, reg, pos, B, Np, R, D, x)
    t = torch.where(masks.unsqueeze(-1), mt.bfloat16().float().unsqueeze(0), tok.float().view(B, Np, D))
    want = torch.cat([cls.expand(B, 1, D), t], 1) + pos
    if R:
        want = torch.cat([want[:, :1], reg.expand(B, R, D), want[:, 1:]], 1)
    torch.testing.assert_close(x, want, rtol=0, atol=1e-6)
    dx = rnd(B, N, D, seed=22)
    dtok = torch.empty(B * Np, D, device=dev, dtype=torch.bfloat16)
    dpos, dcls, dmt = torch.zeros(1 + Np, D, device=dev), torch.zeros(D, device=dev), torch.zeros(D, device=dev)
    dreg = torch.zeros(R, D, device=dev) if R else None
    ops.assemble_tokens_bwd(dx, masks.to(torch.uint8), B, Np, R, D, dtok, dpos, dcls, dreg, dmt)
    dpatch = dx[:, 1 + R:]
    torch.testing.assert_close(dtok.float().view(B, Np, D), torch.where(masks.unsqueeze(-1), torch.zeros(()).to(dev), dpatch).bfloat16().float())
    torch.testing.assert_close(dcls, dx[:, 0].sum(0), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(dpos, torch.cat([dx[:, :1], dpatch], 1).sum(0), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(dmt, (dpatch * masks.unsqueeze(-1)).sum((0, 1)), rtol=1e-5, atol=1e-5)
    if R:
        torch.testing.assert_close(dreg, dx[:, 1:1 + R].sum(0), rtol=1e-5, atol=1e-5)


def test_layerscale_bwd():
    T, D = 999, 384
    dx, o, gamma = rnd(T, D, seed=23), rnd(T, D, dtype=torch.bfloat16, seed=24), rnd(D, seed=25)
    rs = torch.rand(T // 37 + 1, device=dev)
    dout = torch.empty(T, D, device=dev, dtype=torch.bfloat16)
    dg, dbias = torch.zeros(D, device=dev), torch.zeros(D, device=dev)
    ops.layerscale_bwd(dx, o, gamma, rs, 37, dout, dg, dbias)
    g = dx * rs.repeat_interleave(37)[:T, None]
    torch.testing.assert_close(dout.float(), (g * gamma).bfloat16().float())
    torch.testing.assert_close(dg, (g * o.float()).sum(0), rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(dbias, dout.float().sum(0), rtol=1e-4, atol=1e-3)


def test_gather_scatter_rows():
    B, Np, R, D = 4, 36, 4, 128
    N = 1 + R + Np
    src = rnd(B * N, D, seed=26)
    idx = torch.randperm(B * Np, device=dev)[:50].sort().values
    out = torch.empty(50, D, device=dev)
    ops.gather_rows(src, idx, out, Np=Np, N=N, off=1 + R)
    want = src.view(B, N, D)[:, 1 + R:].reshape(B * Np, D)[idx]
    assert torch.equal(out, want)
    outb = torch.empty(50, D, device=dev, dtype=torch.bfloat16)
    ops.gather_rows(src, idx, outb, Np=Np, N=N, off=1 + R)
    assert torch.equal(outb, want.bfloat16())
    dst = torch.zeros(B * N, D, device=dev)
    ops.scatter_rows(out, idx, dst, Np=Np, N=N, off=1 + R)
    ref = torch.zeros(B, N, D, device=dev)
    ref[:, 1 + R:].reshape(B * Np, D)  # view check only
    tmp = torch.zeros(B * Np, D, device=dev); tmp[idx] = out
    ref[:, 1 + R:] = tmp.view(B, Np, D)
    assert torch.equal(dst.view(B, N, D), ref)


def test_l2norm_and_weightnorm():
    R, D = 333, 256
    x = rnd(R, D, dtype=torch.bfloat16, seed=27)
    y, nrm = torch.empty_like(x), torch.empty(R, device=dev)
    ops.l2norm_fwd(x, y, nrm)
    xf = x.float().requires_grad_(True)
    ref = F.normalize(xf, dim=-1, eps=1e-12)
    torch.testing.assert_close(y.float(), ref.bfloat16().float(), rtol=1e-2, atol=1e-2)
    dy = rnd(R, D, dtype=torch.bfloat16, seed=28)
    ref.backward(dy.float())
    dx = torch.empty_like(x)
    ops.l2norm_bwd(dy, x, nrm, dx)
    torch.testing.assert_close(dx.float(), xf.grad, rtol=3e-2, atol=3e-3)
    O, I = 1000, 256
    g, v = (1 + 0.1 * rnd(O, 1, seed=29)).requires_grad_(True), rnd(O, I, seed=30).requires_grad_(True)
    w, vn = torch.empty(O, I, device=dev, dtype=torch.bfloat16), torch.empty(O, device=dev)
    ops.weightnorm_fwd(g.detach(), v.detach(), w, vn)
    wref = g * v / v.norm(dim=1, keepdim=True)
    torch.testing.assert_close(w.float(), wref.bfloat16().float(), rtol=1e-2, atol=1e-3)
    dW = rnd(O, I, seed=31)
    wref.backward(dW)
    dg, dv = torch.zeros(O, 1, device=dev), torch.zeros(O, I, device=dev)
    ops.weightnorm_bwd(dW, g.detach(), v.detach(), dg, dv)
    torch.testing.assert_close(dg, g.grad, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(dv, v.grad, rtol=1e-4, atol=1e-5)


def test_small_matmul_cast_fill():
    A, Bm = rnd(36, 196, seed=32), rnd(196, 384, seed=33)
    Cm = torch.empty(36, 384, device=dev)
    ops.small_matmul(A, Bm, Cm)
    torch.testing.assert_close(Cm, A @ Bm, rtol=1e-4, atol=1e-4)
    G = rnd(36, 384, seed=34)
    Ct = torch.ones(196, 384, device=dev)
    ops.small_matmul(A, G, Ct, a_trans=True, accumulate=True)
    torch.testing.assert_close(Ct, 1 + A.t() @ G, rtol=1e-4, atol=1e-4)
    x = rnd(100003, seed=35)
    y = torch.empty(100003, device=dev, dtype=torch.bfloat16)
    ops.cast_bf16(x, y)
    assert torch.equal(y, x.bfloat16())
    ops.fill_f32(x, 3.0)
    assert torch.equal(x, torch.full_like(x, 3.0))


@pytest.mark.parametrize("K", [65536, 512, 4096 + 8])
def test_loss_kernels(K):
    Rt, Rs = 20, 52
    t = rnd(Rt, K, dtype=torch.bfloat16, seed=36)
    s = rnd(Rs, K, dtype=torch.bfloat16, seed=37)
    center = rnd(K, scale=0.1, seed=38)
    t_scale, s_scale = 1 / 0.05, 10.0
    colterm = torch.empty(K, device=dev)
    ops.vec_op(colterm, center, t_scale, 0.0, 1)
    torch.testing.assert_close(colterm, -center * t_scale)
    rowterm = torch.empty(Rt, device=dev)
    ops.row_lse(t, colterm, t_scale, rowterm)
    z = t.float() * t_scale + colterm
    torch.testing.assert_close(rowterm, -torch.logsumexp(z, -1), rtol=1e-5, atol=1e-4)
    probs = torch.softmax(z, -1)
    i0 = torch.randint(0, Rt, (Rs,), device=dev, dtype=torch.int32)
    i1 = torch.randint(0, Rt, (Rs,), device=dev, dtype=torch.int32)
    i1[::3] = -1
    w = torch.rand(Rs, device=dev)
    loss_rows = torch.empty(Rs, device=dev)
    ds = torch.empty(Rs, K, device=dev, dtype=torch.bfloat16)
    ops.dino_ce(s, t, colterm, rowterm, i0, i1, w, s_scale, t_scale, loss_rows, ds, gscale=2.0)
    sf = s.float().requires_grad_(True)
    lsm = F.log_softmax(sf * s_scale, -1)
    pt = probs[i0.long()] + torch.where((i1 >= 0)[:, None], probs[i1.clamp(min=0).long()], torch.zeros(()).to(dev))
    ref_rows = -(pt * lsm).sum(-1) * w
    torch.testing.assert_close(loss_rows, ref_rows, rtol=1e-4, atol=1e-4)
    (ref_rows.sum() * 2.0).backward()
    err = (ds.float() - sf.grad).abs().max().item()
    assert err <= 1e-2 * sf.grad.abs().max().item() + 1e-8, err
    # single-teacher rows with the teacher log-sum-exp fused into the CE kernel (t_rowterm=None: the iBOT term)
    loss2, ds2 = torch.empty(Rs, device=dev), torch.empty(Rs, K, device=dev, dtype=torch.bfloat16)
    ops.dino_ce(s, t, colterm, None, i0, None, w, s_scale, t_scale, loss2, ds2, gscale=2.0)
    sf2 = s.float().requires_grad_(True)
    ref2 = -(probs[i0.long()] * F.log_softmax(sf2 * s_scale, -1)).sum(-1) * w
    torch.testing.assert_close(loss2, ref2, rtol=1e-4, atol=1e-4)
    (ref2.sum() * 2.0).backward()
    assert (ds2.float() - sf2.grad).abs().max().item() <= 1e-2 * sf2.grad.abs().max().item() + 1e-8
    loss3 = torch.empty(Rs, device=dev)
    ops.dino_ce(s, t, None, None, i0, None, None, s_scale, t_scale, loss3)  # no colterm / weights / gradient
    ref3 = -(torch.softmax(t.float() * t_scale, -1)[i0.long()] * F.log_softmax(s.float() * s_scale, -1)).sum(-1)
    torch.testing.assert_close(loss3, ref3, rtol=1e-4, atol=1e-4)
    # column reductions
    cs = torch.zeros(K, device=dev)
    ops.col_reduce(t, cs)
    torch.testing.assert_close(cs, t.float().sum(0), rtol=1e-4, atol=1e-3)
    rv = rnd(Rt, seed=39)
    cs2 = torch.zeros(K, device=dev)
    ops.col_reduce(t, cs2, rowvec=rv, scale=t_scale, mode=1)
    torch.testing.assert_close(cs2, torch.exp(t.float() * t_scale + rv[:, None]).sum(0), rtol=1e-4, atol=1e-3)
    offs = torch.tensor([0, 10, 30, Rs], device=dev, dtype=torch.int32)
    out = torch.empty(3, device=dev)
    ops.segment_sum(loss_rows, offs, out)
    torch.testing.assert_close(out, torch.stack([loss_rows[:10].sum(), loss_rows[10:30].sum(), loss_rows[30:].sum()]))


@pytest.mark.parametrize("n,D", [(64, 384), (128, 384), (128, 768), (40, 1024), (300, 128)])
def test_koleo(n, D):
    """(64, 384): one CTA per group with the features in shared memory; the other sizes exceed 220 KB of shared memory (or
    256 rows) and take the row-tiled path (ViT-B / ViT-L at large per-GPU batches)."""
    groups = 2
    x = rnd(groups * n, D, seed=40).requires_grad_(True)
    loss = torch.empty(groups, device=dev)
    dx = torch.zeros(groups * n, D, device=dev)
    nn_idx = torch.empty(groups * n, device=dev, dtype=torch.int32)
    ops.koleo(x.detach(), groups, n, loss, dx, gscale=0.1, bf16_sim=False, nn_out=nn_idx)
    tot = 0
    for gI in range(groups):
        xn = F.normalize(x[gI * n:(gI + 1) * n], p=2, dim=-1, eps=1e-8)
        sim = (xn @ xn.t()).detach().clone()
        sim.fill_diagonal_(-2)
        idx = sim.argmax(1)
        assert torch.equal(idx.int(), nn_idx[gI * n:(gI + 1) * n])
        d = F.pairwise_distance(xn, xn[idx], p=2.0, eps=1e-8)
        l = -(d + 1e-8).log().mean()
        torch.testing.assert_close(loss[gI], l, rtol=1e-5, atol=1e-5)
        tot = tot + l
    (0.1 * tot).backward()
    torch.testing.assert_close(dx, x.grad, rtol=1e-3, atol=1e-6)


def test_ema_sumsq_adamw():
    n = 1024 * 38
    t, s = rnd(n, seed=41), rnd(n, seed=42)
    tb = torch.empty(n, device=dev, dtype=torch.bfloat16)
    want = t * 0.25 + s * 0.75
    ops.ema(t, s, 0.25, tb)
    torch.testing.assert_close(t, want, rtol=0, atol=1e-7)
    assert torch.equal(tb, t.bfloat16())
    ss = torch.zeros(1, device=dev)
    ops.sumsq(s, ss)
    torch.testing.assert_close(ss[0], (s.double() ** 2).sum().float(), rtol=1e-5, atol=0)
    # fused clip + AdamW + EMA vs torch.optim.AdamW on two groups
    p = rnd(n, seed=43); g = rnd(n, seed=44) * 3; teacher = rnd(n, seed=45)
    p_ref = p.clone().requires_grad_(True)
    half = n // 2
    pa, pb = p_ref[:half].detach().clone().requires_grad_(True), p_ref[half:].detach().clone().requires_grad_(True)
    opt = torch.optim.AdamW([{"params": [pa], "lr": 1e-2, "weight_decay": 0.04},
                             {"params": [pb], "lr": 1e-2 * 0.5, "weight_decay": 0.0}], betas=(0.9, 0.999), eps=1e-8)
    m_, v_ = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    pb16, tb16 = torch.empty(n, device=dev, dtype=torch.bfloat16), torch.empty(n, device=dev, dtype=torch.bfloat16)
    lr_scale = torch.ones(n // 1024, device=dev); lr_scale[half // 1024:] = 0.5
    wd_scale = torch.ones(n // 1024, device=dev); wd_scale[half // 1024:] = 0.0
    t_ref = teacher.clone()
    for step in (1, 2, 3):
        gs = g * step
        pa.grad, pb.grad = gs[:half].clone(), gs[half:].clone()
        torch.nn.utils.clip_grad_norm_([pa, pb], 3.0)
        opt.step()
        t_ref = t_ref * 0.9 + torch.cat([pa, pb]).detach() * 0.1
        nsq = torch.zeros(1, device=dev)
        ops.sumsq(gs, nsq)
        a = ops.AdamWArgs()
        a.p, a.g, a.m, a.v, a.t = p.data_ptr(), gs.data_ptr(), m_.data_ptr(), v_.data_ptr(), teacher.data_ptr()
        a.p_bf16, a.t_bf16 = pb16.data_ptr(), tb16.data_ptr()
        a.n, a.chunk = n, 1024
        a.lr_scale, a.wd_scale, a.flags = lr_scale.data_ptr(), wd_scale.data_ptr(), None
        a.lr, a.wd, a.beta1, a.beta2, a.eps, a.step, a.ema_m = 1e-2, 0.04, 0.9, 0.999, 1e-8, step, 0.9
        a.gradnorm_sq, a.max_norm, a.grad_scale = nsq.data_ptr(), 3.0, 1.0
        ops.adamw_ema(a)
        torch.testing.assert_close(p, torch.cat([pa, pb]).detach(), rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(teacher, t_ref, rtol=1e-5, atol=1e-6)
    assert torch.equal(pb16, p.bfloat16()) and torch.equal(tb16, teacher.bfloat16())


@pytest.mark.parametrize("T,H", [(1000, 344), (77, 2048), (5, 8)])
def test_swiglu_gate_fwd_bwd(T, H):
    """b200_swiglu_fwd/bwd vs torch on bf16 tensors (the autocast reference: silu and the product each round to bf16)."""
    x12 = rnd(T, 2 * H, dtype=torch.bfloat16, scale=2.0, seed=31)
    hid = torch.empty(T, H, device=dev, dtype=torch.bfloat16)
    ops.swiglu_fwd(x12, hid)
    xr = x12.clone().requires_grad_(True)
    x1, x2 = xr.chunk(2, dim=-1)
    want = F.silu(x1) * x2
    torch.testing.assert_close(hid.float(), want.float(), rtol=1.6e-2, atol=1e-3)  # <= 2 bf16 ulp (rcp/ex2.approx sigmoid)
    dh = rnd(T, H, dtype=torch.bfloat16, scale=1.0, seed=32)
    want.backward(dh)
    dx = torch.empty_like(x12)
    ops.swiglu_bwd(x12, dh, dx)
    torch.testing.assert_close(dx.float(), xr.grad.float(), rtol=2.4e-2, atol=2e-3)
    rel = (dx.float() - xr.grad.float()).norm() / xr.grad.float().norm()
    assert rel < 5e-3, rel


@pytest.mark.parametrize("n,k", [(64, 51), (128, 89), (512, 358), (2048, 1433), (5, 1)])
def test_random_subset(n, k):
    """b200_random_subset vs the definition it replaces (torch.randperm(n)[:k], block.py:125-127): k distinct indices in
    range, a fresh draw per launch (device-side counter), every element included with probability k / n."""
    counter = torch.zeros(1, device=dev, dtype=torch.int64)
    hits = torch.zeros(n, device=dev)
    first = torch.zeros(n, device=dev)
    prev = None
    reps = 400
    for i in range(reps):
        idx = torch.empty(k, device=dev, dtype=torch.int64)
        ops.random_subset(n, k, 1234, counter, idx)
        assert int(idx.min()) >= 0 and int(idx.max()) < n and idx.unique().numel() == k
        if prev is not None and k < n and n > 8:
            assert not torch.equal(prev, idx)
        prev = idx
        hits[idx] += 1
        first[idx[0]] += 1
    assert int(counter) == reps
    p = k / n
    tol = 5 * (p * (1 - p) / reps) ** 0.5 + 1e-9
    assert (hits / reps - p).abs().max().item() < tol                      # inclusion probability
    if n >= 64:
        assert first.max().item() < reps * (1.0 / n) + 6 * (reps / n) ** 0.5 + 2  # the leading element is uniform too
    # same seed + same counter -> same subset (reproducibility under torch.manual_seed in the model)
    c2 = torch.zeros(1, device=dev, dtype=torch.int64)
    a = torch.empty(k, device=dev, dtype=torch.int64); ops.random_subset(n, k, 99, c2, a)
    c3 = torch.zeros(1, device=dev, dtype=torch.int64)
    b = torch.empty(k, device=dev, dtype=torch.int64); ops.random_subset(n, k, 99, c3, b)
    assert torch.equal(a, b)


@pytest.mark.parametrize("M,K,N,epi,bn", [(1000, 384, 1152, "bf16", 0), (1000, 384, 1152, "bf16", 192), (300, 192, 576, "bf16", 0),
                                          (1000, 384, 1536, "gelu", 0), (1000, 384, 1536, "gelu_dg", 0), (129, 384, 1536, "gelu_dg", 128),
                                          (18944, 384, 1152, "bf16", 0)])
def test_ln_gemm_prologue(M, K, N, epi, bn):
    """b200_ln_gemm (LayerNorm as the GEMM's A-operand prologue) against the two-kernel path it replaces (b200_layernorm_fwd
    -> b200_gemm) and against torch: same normalised rows (bit-exact side outputs), same GEMM result up to accumulation order."""
    x = rnd(M, K, scale=2.0, seed=40) + 0.3
    lw, lb = 1.0 + rnd(K, scale=0.2, seed=41), rnd(K, scale=0.1, seed=42)
    w = rnd(N, K, dtype=torch.bfloat16, scale=0.05, seed=43)
    bias = rnd(N, scale=0.1, seed=44)
    code = {"bf16": ops.EPI_BF16, "gelu": ops.EPI_BIAS_GELU, "gelu_dg": ops.EPI_BIAS_GELU_DG}[epi]
    # two-kernel reference
    xn_ref = torch.empty(M, K, device=dev, dtype=torch.bfloat16)
    mean_ref, rstd_ref = torch.empty(M, device=dev), torch.empty(M, device=dev)
    ops.layernorm_fwd(x, lw, lb, 1e-6, xn_ref, mean_ref, rstd_ref)
    out_ref = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    out2_ref = torch.empty(M, N, device=dev, dtype=torch.bfloat16) if epi == "gelu_dg" else None
    ops.gemm(xn_ref, w, out_ref, epi=code, bias=bias, out2=out2_ref)
    # fused
    xn = torch.full((M, K), 7.0, device=dev, dtype=torch.bfloat16)
    mean, rstd = torch.empty(M, device=dev), torch.empty(M, device=dev)
    out = torch.full((M, N), 7.0, device=dev, dtype=torch.bfloat16)
    out2 = torch.full((M, N), 7.0, device=dev, dtype=torch.bfloat16) if epi == "gelu_dg" else None
    ops.ln_gemm(x, lw, lb, 1e-6, w, out, epi=code, bias=bias, out2=out2, xn_out=xn, mean=mean, rstd=rstd, block_n=bn)
    torch.cuda.synchronize()
    assert torch.equal(xn, xn_ref) and torch.equal(mean, mean_ref) and torch.equal(rstd, rstd_ref)
    torch.testing.assert_close(out.float(), out_ref.float(), rtol=1.6e-2, atol=2e-3)  # <= 2 bf16 ulp
    assert (out.float() - out_ref.float()).abs().mean().item() < 1e-4
    if out2 is not None:
        torch.testing.assert_close(out2.float(), out2_ref.float(), rtol=1.6e-2, atol=2e-3)
    # without the side outputs (teacher / recompute): same product
    out_b = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    ops.ln_gemm(x, lw, lb, 1e-6, w, out_b, epi=code, bias=bias, block_n=bn)
    assert torch.equal(out_b, out)
    # torch statement (fp32 LayerNorm, bf16-rounded activations and weights, fp32 accumulate)
    y = torch.nn.functional.layer_norm(x, (K,), lw, lb, 1e-6).bfloat16().float() @ w.float().t() + bias
    if epi != "bf16":
        y = torch.nn.functional.gelu(y.bfloat16().float())
    torch.testing.assert_close(out.float(), y, rtol=2e-2, atol=2e-2)
