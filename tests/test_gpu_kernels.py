"""GPU: every C-ABI kernel against the oracle / an fp64 evaluation of the same operands.

Tolerances: integer outputs (argmax, matches) are bit-exact; fp32 kernels 1e-4..1e-5 relative;
bf16 tensor-core kernels are compared with an fp64 evaluation of the SAME bf16-rounded operands, so
the only difference is fp32 accumulation order and the bf16 rounding of the softmax probabilities
(2^-9 relative per element) -> 1e-2 on outputs/gradients is the stated tolerance there.
"""
import math
import os

import numpy as np
import pytest
import torch

from gluefactory_b200 import ops
from oracle import lightglue_oracle as O
from tests.util import GOLDEN, load_gluestick_attn, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _rand(*shape, seed=0, dtype=torch.float32, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(dtype).to(DEV)


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("shape", [(2, 256, 256, 256), (3, 200, 136, 72), (1, 128, 128, 64), (2, 384, 64, 512)])
def test_gemm_bf16_tcgen05(a_mn, b_mn, shape):
    batch, M, N, K = shape
    a = _rand(batch, K, M, seed=1, dtype=torch.bfloat16) if a_mn else _rand(batch, M, K, seed=1, dtype=torch.bfloat16)
    b = _rand(batch, K, N, seed=2, dtype=torch.bfloat16) if b_mn else _rand(batch, N, K, seed=2, dtype=torch.bfloat16)
    A = a.double().transpose(1, 2) if a_mn else a.double()
    Bm = b.double().transpose(1, 2) if b_mn else b.double()
    ref = A @ Bm.transpose(1, 2)
    c = ops.gemm_bf16(a, b, bool(a_mn), bool(b_mn), out_dtype=torch.float32)
    assert rel_err(c, ref) < 1e-5
    c16 = ops.gemm_bf16(a, b, bool(a_mn), bool(b_mn), out_dtype=torch.bfloat16)
    assert rel_err(c16, ref) < 4e-3


@pytest.mark.parametrize("T,M,N", [(4096, 256, 256), (10000, 512, 256), (777, 768, 256), (300, 256, 512), (64, 128, 72)])
def test_wgrad_splitk(T, M, N):
    """dW = dy^T a (autograd of F.linear) through the split-K tcgen05 GEMM, both operands MN-major as stored."""
    dy = _rand(T, M, seed=1, dtype=torch.bfloat16)
    a = _rand(T, N, seed=2, dtype=torch.bfloat16)
    ref = dy.double().t() @ a.double()
    w1 = ops.wgrad_bf16(dy, a)
    assert rel_err(w1, ref) < 1e-5
    assert torch.equal(w1, ops.wgrad_bf16(dy, a))  # fixed summation order
    # strided operand views (column slices of wider activations), as the layer backward passes them
    wide = _rand(T, 2 * N, seed=3, dtype=torch.bfloat16)
    assert rel_err(ops.wgrad_bf16(dy, wide[:, N:]), dy.double().t() @ wide[:, N:].double()) < 1e-5


@pytest.mark.parametrize("T,K,N", [(4096, 256, 768), (1000, 512, 512), (777, 512, 256), (130, 256, 256), (64, 128, 72)])
def test_linear_epilogues(T, K, N):
    """lgb200_linear: y = x W^T + b with the fp32 bias added in the epilogue, into a column block of a wider matrix;
    dx = dy W (W read as stored); fp32 accumulate-into-dx through the TMA reduce."""
    wide = _rand(T, 2 * K, seed=1, dtype=torch.bfloat16)
    x = wide[:, K:]                                   # row-strided A (the [x | msg] FFN input halves)
    w = _rand(N, K, seed=2, dtype=torch.bfloat16, scale=K ** -0.5)
    b = _rand(N, seed=3)
    ref = x.double() @ w.double().t() + b.double()
    y = ops.linear(x, w, b)
    assert y.dtype == torch.bfloat16 and rel_err(y, ref) < 4e-3
    y32 = ops.linear(x, w, b, out_dtype=torch.float32)
    assert rel_err(y32, ref) < 1e-5
    if N % 8 == 0:
        out_wide = torch.zeros(T, 2 * N, device=DEV, dtype=torch.bfloat16)
        ops.linear(x, w, b, out=out_wide[:, N:])          # row-strided C
        assert rel_err(out_wide[:, N:], ref) < 4e-3 and float(out_wide[:, :N].abs().sum()) == 0.0
    # dgrad: dy [T, N] @ W [N, K] (B operand MN-major, exactly as the weight lies in memory)
    dy = _rand(T, N, seed=4, dtype=torch.bfloat16)
    refdx = dy.double() @ w.double()
    assert rel_err(ops.linear(dy, w, w_is_kn=True), refdx) < 4e-3
    if K % 4 == 0:
        acc0 = _rand(T, K, seed=5)
        acc = acc0.clone()
        ops.linear(dy, w, out=acc, w_is_kn=True, accumulate=True)
        assert rel_err(acc, acc0.double() + refdx) < 1e-5
        # a column slice of a wider weight (ffn.0's [x | msg] halves)
        wwide = _rand(N, 2 * K, seed=6, dtype=torch.bfloat16, scale=K ** -0.5)
        acc = acc0.clone()
        ops.linear(dy, wwide[:, K:], out=acc, w_is_kn=True, accumulate=True)
        assert rel_err(acc, acc0.double() + dy.double() @ wwide[:, K:].double()) < 1e-5


def test_linear_autograd_function():
    x = _rand(515, 256, seed=1, dtype=torch.bfloat16).requires_grad_(True)
    lin = torch.nn.Linear(256, 384).to(DEV)
    y = ops.LinearFn.apply(x, lin.weight, lin.bias)
    g = _rand(515, 384, seed=2, dtype=torch.bfloat16)
    y.backward(g)
    xr = x.detach().double().requires_grad_(True)
    wr = lin.weight.detach().to(torch.bfloat16).double().requires_grad_(True)
    br = lin.bias.detach().double().requires_grad_(True)
    (xr @ wr.t() + br).backward(g.double())
    assert rel_err(x.grad, xr.grad) < 4e-3
    assert rel_err(lin.weight.grad, wr.grad) < 1e-5 and rel_err(lin.bias.grad, br.grad) < 1e-5


@pytest.mark.parametrize("B,M,N,D", [(2, 256, 256, 256), (3, 150, 203, 256), (1, 72, 300, 128), (2, 2048, 2048, 256),
                                     (1, 130, 64, 64)])
def test_assign_fused_matches_unfused_and_fp64(B, M, N, D):
    """csrc/assign_tc.cu (similarity never leaves tensor memory) against (a) the round-1 path -- sim GEMM written to HBM,
    assign_lse / assign_scores / assign_bwd, two d(mdesc) GEMMs -- and (b) an fp64 evaluation of the same bf16 operands."""
    md0 = _rand(B, M, D, seed=1, dtype=torch.bfloat16, scale=2.0)
    md1 = _rand(B, N, D, seed=2, dtype=torch.bfloat16, scale=2.0)
    alpha = D ** -0.5
    z0, z1 = _rand(B, M, seed=3), _rand(B, N, seed=4)
    ls0, ls1 = torch.nn.functional.logsigmoid(z0), torch.nn.functional.logsigmoid(z1)
    du0, du1 = torch.nn.functional.logsigmoid(-z0), torch.nn.functional.logsigmoid(-z1)
    g = torch.Generator().manual_seed(5)
    gt = torch.zeros(B, M, N, dtype=torch.bool)
    K = min(M, N) // 3
    for b in range(B):
        gt[b, torch.randperm(M, generator=g)[:K], torch.randperm(N, generator=g)[:K]] = True
    gt = gt.to(DEV)
    gt_u8 = gt.view(torch.uint8)
    f = ops.assign_fused_stats(md0, md1, alpha, ls0, ls1, gt_u8=gt_u8)
    sim = ops.gemm_bf16(md0, md1, alpha=alpha)
    u = ops.assign_stats(sim, ls0, ls1, du0, du1, gt_u8=gt_u8, dense=False)
    # (a) same fp32 accumulators, different summation grouping in the LSE: 1e-5; integer outputs equal
    for k in ("lse_row", "lse_col", "rowmax", "colmax"):
        assert (f[k] - u[k]).abs().max().item() < 2e-4, k
    same_r = (f["rowarg"] == u["rowarg"]).float().mean().item()
    same_c = (f["colarg"] == u["colarg"]).float().mean().item()
    assert same_r > 0.999 and same_c > 0.999, (same_r, same_c)  # argmax flips only on fp32-rounding near-ties
    assert (f["pos_row_sum"] - u["pos_row_sum"]).abs().max().item() < 1e-3
    # (b) fp64 on the same bf16 operands
    s64 = (md0.double() @ md1.double().transpose(1, 2)) * alpha
    assert (f["lse_row"].double() - torch.logsumexp(s64, 2)).abs().max().item() < 1e-4
    assert (f["lse_col"].double() - torch.logsumexp(s64, 1)).abs().max().item() < 1e-4
    sc = (s64 - torch.logsumexp(s64, 2, keepdim=True)) + (s64 - torch.logsumexp(s64, 1, keepdim=True)) + \
        (ls0.double()[:, :, None] + ls1.double()[:, None, :])
    assert (f["rowmax"].double() - sc.max(2).values).abs().max().item() < 1e-3
    assert (f["colmax"].double() - sc.max(1).values).abs().max().item() < 1e-3
    # backward
    rowcnt, colcnt = gt_u8.sum(2, dtype=torch.float32), gt_u8.sum(1, dtype=torch.float32)
    gc = (_rand(B, seed=6).abs() + 0.1) * alpha
    dmd = torch.empty(B * M + B * N, D, device=DEV, dtype=torch.bfloat16)
    ops.assign_fused_bwd(md0, md1, alpha, f["lse_row"], f["lse_col"], gt_u8, gt_u8.transpose(1, 2).contiguous(), gc, rowcnt,
                         colcnt, dmd[:B * M], dmd[B * M:])
    p_r = torch.exp(s64 - torch.logsumexp(s64, 2, keepdim=True))
    p_c = torch.exp(s64 - torch.logsumexp(s64, 1, keepdim=True))
    dsim = gc.double()[:, None, None] * (2 * gt.double() - p_r * rowcnt.double()[:, :, None] - p_c * colcnt.double()[:, None, :])
    ref0 = (dsim @ md1.double()).reshape(B * M, D)
    ref1 = (dsim.transpose(1, 2) @ md0.double()).reshape(B * N, D)
    assert rel_err(dmd[:B * M], ref0) < 8e-3 and rel_err(dmd[B * M:], ref1) < 8e-3  # dsim and the output are bf16
    torch.cuda.synchronize()


def test_gemm_unaligned_output_uses_fallback_epilogue():
    """N = 130: C rows are not 16-byte multiples, so the TMA-store epilogue is replaced by plain stores."""
    a = _rand(2, 100, 64, seed=1, dtype=torch.bfloat16)
    b = _rand(2, 130, 64, seed=2, dtype=torch.bfloat16)
    ref = a.double() @ b.double().transpose(1, 2)
    assert rel_err(ops.gemm_bf16(a, b, alpha=0.5), 0.5 * ref) < 1e-5
    assert rel_err(ops.gemm_bf16(a, b, out_dtype=torch.bfloat16), ref) < 4e-3


# ------------------------------------------------------------------------------------------------
def _attn_ref(q, k, v, shift):
    """fp64 attention on [B,N,H,64] with the kv batch roll."""
    q, k, v = (t.double().permute(0, 2, 1, 3) for t in (q, k, v))
    B = q.shape[0]
    idx = (torch.arange(B, device=q.device) + shift) % B
    k, v = k[idx], v[idx]
    s = q @ k.transpose(-1, -2) / 8.0
    return (torch.softmax(s, -1) @ v).permute(0, 2, 1, 3), torch.logsumexp(s, -1)


ATTN_SHAPES = [(2, 128, 128, 4, 0), (2, 256, 256, 4, 1), (2, 200, 200, 2, 1), (1, 72, 300, 4, 0), (4, 512, 512, 4, 2)]


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 2e-5), (torch.bfloat16, 1e-2)])
@pytest.mark.parametrize("B,Nq,Nk,H,shift", ATTN_SHAPES)
def test_attention_forward_backward(dtype, tol, B, Nq, Nk, H, shift):
    if shift and Nq != Nk:
        pytest.skip("shifted launch needs equal lengths")
    q = _rand(B, Nq, H, 64, seed=1, dtype=dtype, scale=1.5).requires_grad_(True)
    k = _rand(B, Nk, H, 64, seed=2, dtype=dtype, scale=1.5).requires_grad_(True)
    v = _rand(B, Nk, H, 64, seed=3, dtype=dtype).requires_grad_(True)
    go = _rand(B, Nq, H, 64, seed=4, dtype=dtype)
    out = ops.Attention.apply(q, k, v, shift, 0.125)
    out.backward(go)
    qr, kr, vr = (t.detach().double().requires_grad_(True) for t in (q, k, v))
    ref, _ = _attn_ref(qr, kr, vr, shift)
    ref.backward(go.double())
    assert rel_err(out, ref) < tol
    assert rel_err(q.grad, qr.grad) < tol
    assert rel_err(k.grad, kr.grad) < tol
    assert rel_err(v.grad, vr.grad) < tol


@pytest.mark.parametrize("B,Nq,Nk,H,shift", ATTN_SHAPES)
def test_attention_tc_matches_simt_lse(B, Nq, Nk, H, shift):
    """the tcgen05 forward and the CUDA-core forward must agree on out and on the saved log-sum-exp"""
    from gluefactory_b200._lib import BF16, call, ptr, stream_ptr

    if shift and Nq != Nk:
        pytest.skip("shifted launch needs equal lengths")
    q = _rand(B, Nq, H, 64, seed=1, dtype=torch.bfloat16, scale=1.5)
    k = _rand(B, Nk, H, 64, seed=2, dtype=torch.bfloat16, scale=1.5)
    v = _rand(B, Nk, H, 64, seed=3, dtype=torch.bfloat16)
    out = torch.empty_like(q)
    lse = torch.empty(B, H, Nq, device=DEV)
    call("lgb200_attn_fwd", ptr(q), ptr(k), ptr(v), ptr(out), ptr(lse), B, Nq, Nk, H, shift, 0.125, BF16, stream_ptr())
    ref, ref_lse = _attn_ref(q, k, v, shift)
    assert rel_err(out, ref) < 1e-2
    assert (lse.double() - ref_lse).abs().max().item() < 2e-3


@pytest.mark.parametrize("B,Nq,Nk,H,shift", [(2, 512, 512, 4, 1), (2, 300, 200, 4, 0)])
def test_attention_two_kernel_backward_agrees_with_fused(B, Nq, Nk, H, shift, monkeypatch):
    """The round-1 pair of backward kernels (dQ, dK/dV; deterministic summation order) stays selectable with
    LGB200_ATTN_BWD_TWO_KERNEL=1 as an independent cross-check of the fused single-pass backward."""
    q = _rand(B, Nq, H, 64, seed=1, dtype=torch.bfloat16, scale=1.5)
    k = _rand(B, Nk, H, 64, seed=2, dtype=torch.bfloat16, scale=1.5)
    v = _rand(B, Nk, H, 64, seed=3, dtype=torch.bfloat16)
    go = _rand(B, Nq, H, 64, seed=4, dtype=torch.bfloat16)
    out, lse = ops.attn_fwd(q, k, v, shift, 0.125)
    fused = ops.attn_bwd(q, k, v, out, lse, go, shift, 0.125)
    monkeypatch.setenv("LGB200_ATTN_BWD_TWO_KERNEL", "1")
    two = ops.attn_bwd(q, k, v, out, lse, go, shift, 0.125)
    monkeypatch.delenv("LGB200_ATTN_BWD_TWO_KERNEL")
    for a, b, name in zip(fused, two, ("dq", "dk", "dv")):
        assert rel_err(a, b.double()) < 6e-3, name


def test_linear_generic_kernel_agrees_with_panel_resident(monkeypatch):
    """K <= 256 projections run on the A-panel-resident GEMM by default; LGB200_GEMM_NO_APANEL=1 sends them through the
    generic persistent kernel: same products, same accumulation -> identical results."""
    a = _rand(3000, 256, seed=11, dtype=torch.bfloat16)
    w = _rand(768, 256, seed=12, dtype=torch.bfloat16, scale=0.1)
    bias = _rand(768, seed=13)
    y0 = ops.linear(a, w, bias)
    monkeypatch.setenv("LGB200_GEMM_NO_APANEL", "1")
    y1 = ops.linear(a, w, bias)
    monkeypatch.delenv("LGB200_GEMM_NO_APANEL")
    assert torch.equal(y0, y1)


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-6), (torch.bfloat16, 8e-3)])
def test_rope_split(dtype, tol):
    T, H = 333, 4
    qkv = _rand(T, H * 192, seed=1, dtype=dtype).requires_grad_(True)
    theta = _rand(T, 32, seed=2, scale=3.0).requires_grad_(True)
    q, k, v = ops.RopeSplit.apply(qkv, theta, H)
    gq, gk, gv = (_rand(T, H * 64, seed=s, dtype=dtype) for s in (3, 4, 5))
    torch.autograd.backward([q, k, v], [gq, gk, gv])
    # oracle: lightglue.py:157-160 + 42-49
    x = qkv.detach().double().requires_grad_(True)
    th = theta.detach().double().requires_grad_(True)
    t = x.view(1, T, H, 64, 3).permute(0, 2, 1, 3, 4)
    rq, rk, rv = O.rope(t[..., 0], th[None]), O.rope(t[..., 1], th[None]), t[..., 2]
    back = lambda z: z.permute(0, 2, 1, 3).reshape(T, H * 64)  # noqa: E731
    torch.autograd.backward([back(rq), back(rk), back(rv)], [gq.double(), gk.double(), gv.double()])
    assert rel_err(q, back(rq)) < tol and rel_err(k, back(rk)) < tol and rel_err(v, back(rv)) < tol
    assert rel_err(qkv.grad, x.grad) < tol
    assert rel_err(theta.grad, th.grad) < (1e-5 if dtype == torch.float32 else 2e-2)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 2e-6), (torch.bfloat16, 8e-3)])
@pytest.mark.parametrize("W", [256, 512])
def test_ln_gelu(dtype, tol, W):
    T = 1001
    x = _rand(T, W, seed=1, dtype=dtype, scale=2.0).requires_grad_(True)
    g = (1 + 0.1 * _rand(W, seed=2)).requires_grad_(True)
    b = (0.1 * _rand(W, seed=3)).requires_grad_(True)
    gy = _rand(T, W, seed=4, dtype=dtype)
    y = ops.LnGelu.apply(x, g, b, 1e-5)
    y.backward(gy)
    xr, gr, br = (t.detach().double().requires_grad_(True) for t in (x, g, b))
    ref = torch.nn.functional.gelu(torch.nn.functional.layer_norm(xr, (W,), gr, br, 1e-5))
    ref.backward(gy.double())
    assert rel_err(y, ref) < tol
    assert rel_err(x.grad, xr.grad) < tol
    assert rel_err(g.grad, gr.grad) < max(tol, 1e-5) and rel_err(b.grad, br.grad) < max(tol, 1e-5)


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,M,N", [(2, 96, 96), (1, 80, 112), (2, 257, 130), (1, 1024, 1024), (3, 33, 515)])
def test_assignment_head_matches_oracle(B, M, N):
    sim = _rand(B, M, N, seed=1, scale=4.0)
    z0, z1 = _rand(B, M, seed=2, scale=2.0), _rand(B, N, seed=3, scale=2.0)
    gt = (torch.rand(B, M, N, generator=torch.Generator().manual_seed(4)) < 0.01).to(DEV)
    ls = torch.nn.functional.logsigmoid
    st = ops.assign_stats(sim, ls(z0), ls(z1), ls(-z0), ls(-z1), gt_u8=gt.view(torch.uint8), dense=True)
    ref = O.sigmoid_log_double_softmax(sim.double().cpu(), z0.double().cpu(), z1.double().cpu())
    scores = st["scores"].cpu()
    np.testing.assert_allclose(scores.numpy(), ref.numpy(), rtol=0, atol=2e-5)
    np.testing.assert_allclose(st["lse_row"].cpu().numpy(), torch.logsumexp(sim.double(), 2).cpu().numpy(), atol=1e-5)
    np.testing.assert_allclose(st["lse_col"].cpu().numpy(), torch.logsumexp(sim.double(), 1).cpu().numpy(), atol=1e-5)
    # argmax: bit-exact against torch's max on the kernel's own fp32 scores (ties -> lowest index)
    inner = scores[:, :-1, :-1]
    assert torch.equal(st["rowarg"].cpu().long(), inner.max(2).indices)
    assert torch.equal(st["colarg"].cpu().long(), inner.max(1).indices)
    assert torch.equal(st["rowmax"].cpu(), inner.max(2).values)
    assert torch.equal(st["colmax"].cpu(), inner.max(1).values)
    # ... and against the fp64 oracle wherever its top-2 margin exceeds fp32 resolution
    top2 = ref[:, :-1, :-1].topk(2, dim=2).values
    safe = (top2[..., 0] - top2[..., 1]) > 1e-4
    assert torch.equal(st["rowarg"].cpu().long()[safe], ref[:, :-1, :-1].max(2).indices[safe])
    # filter_matches
    for th in (0.0, 0.05):
        m0, m1, ms0, ms1 = ops.filter_matches(st["rowmax"], st["rowarg"], st["colarg"], th)
        r0, r1, rs0, rs1 = O.filter_matches(scores, th)
        assert torch.equal(m0.cpu(), r0) and torch.equal(m1.cpu(), r1)
        np.testing.assert_allclose(ms0.cpu().numpy(), rs0.numpy(), rtol=1e-6)
        np.testing.assert_allclose(ms1.cpu().numpy(), rs1.numpy(), rtol=1e-6)
    # positive-weighted sum and row_norm monitor
    pos_ref = ((2 * sim.double() - torch.logsumexp(sim.double(), 2, keepdim=True)
                - torch.logsumexp(sim.double(), 1, keepdim=True)) * gt).sum(2)
    np.testing.assert_allclose(st["pos_row_sum"].cpu().numpy(), pos_ref.cpu().numpy(), rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(st["row_expsum"].cpu().numpy(), ref.exp()[:, :-1].sum(2).numpy(), rtol=1e-4)


@pytest.mark.parametrize("bf16", [False, True])
@pytest.mark.parametrize("B,M,N", [(2, 128, 128), (1, 200, 136), (2, 100, 250)])
def test_assign_positives_backward(bf16, B, M, N):
    D = 256
    md0 = _rand(B, M, D, seed=1, scale=0.3).requires_grad_(True)
    md1 = _rand(B, N, D, seed=2, scale=0.3).requires_grad_(True)
    z0, z1 = _rand(B, M, seed=3), _rand(B, N, seed=4)
    gt = (torch.rand(B, M, N, generator=torch.Generator().manual_seed(5)) < 0.02).to(DEV)
    ls = torch.nn.functional.logsigmoid
    s_pos, *_ = ops.AssignPositives.apply(md0, md1, ls(z0), ls(z1), ls(-z0), ls(-z1), gt.view(torch.uint8),
                                          gt.sum(2).float(), gt.sum(1).float(), bf16)
    gw = _rand(B, seed=6)
    (s_pos * gw).sum().backward()
    rnd = O.bf16_round if bf16 else (lambda t: t)
    a, b = rnd(md0.detach()).double().requires_grad_(True), rnd(md1.detach()).double().requires_grad_(True)
    sim = a @ b.transpose(1, 2)
    ref = ((2 * sim - torch.logsumexp(sim, 2, keepdim=True) - torch.logsumexp(sim, 1, keepdim=True)) * gt).sum((1, 2))
    (ref * gw.double()).sum().backward()
    tol = 2e-2 if bf16 else 1e-4
    assert rel_err(s_pos, ref) < (1e-3 if bf16 else 1e-5)
    assert rel_err(md0.grad, a.grad) < tol and rel_err(md1.grad, b.grad) < tol


def test_other_heads_match_golden():
    g = dict(np.load(os.path.join(GOLDEN, "heads.npz")))
    for tag in ["a", "b"]:
        sim = torch.from_numpy(g[f"{tag}|sim"]).float().to(DEV)
        np.testing.assert_allclose(ops.log_double_softmax(sim, 0.7).cpu().numpy(), g[f"{tag}|lds"], atol=2e-5)
        np.testing.assert_allclose(ops.log_optimal_transport(sim, 0.7, 50).cpu().numpy(), g[f"{tag}|lot"], atol=1e-4)


def test_other_heads_backward_matches_reference_autograd():
    """GlueStick / SuperGlue heads are differentiable (forward kernels + heads_grad.py): gradients w.r.t. the
    similarity and the bin score against the reference's autograd (tests/golden/heads_grad.npz)."""
    g = dict(np.load(os.path.join(GOLDEN, "heads_grad.npz")))
    for tag in ["a", "b"]:
        w = torch.from_numpy(g[f"{tag}|w"]).float().to(DEV)
        for name, fn in (("lds", lambda s_, b_: ops.log_double_softmax(s_, b_)),
                         ("lot", lambda s_, b_: ops.log_optimal_transport(s_, b_, 50))):
            sim = torch.from_numpy(g[f"{tag}|sim"]).float().to(DEV).requires_grad_()
            beta = torch.tensor(0.7, device=DEV, requires_grad=True)
            (fn(sim, beta) * w).sum().backward()
            assert rel_err(sim.grad, torch.from_numpy(g[f"{tag}|{name}|dsim"])) < 1e-3, (tag, name)
            ref = float(g[f"{tag}|{name}|dbin"])
            assert abs(beta.grad.item() - ref) < 1e-3 * max(1.0, abs(ref)), (tag, name, beta.grad.item(), ref)


@pytest.mark.parametrize("B,M,N,iters", [(1, 2048, 2048, 50), (2, 2048, 2048, 20), (3, 1000, 777, 50),
                                          (160, 40, 56, 10), (1, 3, 5, 1), (2, 130, 97, 0)])
def test_sinkhorn_kernels_at_size(B, M, N, iters):
    """Persistent Sinkhorn forward + reverse-sweep backward (csrc/heads.cu) against fp64 autograd through the
    restated iterations (superglue.py:186-214) at the benchmark size (strip cache path), without the cache (B=2),
    ragged shapes, more pairs than SMs, tiny and zero-iteration cases."""
    from gluefactory_b200 import heads_grad

    sim = (_rand(B, M, N, seed=31) * 3.0).requires_grad_()
    alpha = torch.tensor(0.9, device=DEV, requires_grad=True)
    w = _rand(B, M + 1, N + 1, seed=32)
    out = ops.log_optimal_transport(sim, alpha, iters)
    (out * w).sum().backward()
    sd = sim.detach().double().requires_grad_()
    ad = alpha.detach().double().requires_grad_()
    Z = torch.cat([torch.cat([sd, ad.expand(B, M, 1)], 2), ad.expand(B, 1, N + 1)], 1)
    norm = -np.log(M + N)
    log_mu = torch.full((B, M + 1), norm, device=DEV, dtype=torch.float64)
    log_mu[:, M] += np.log(N)
    log_nu = torch.full((B, N + 1), norm, device=DEV, dtype=torch.float64)
    log_nu[:, N] += np.log(M)
    u, v = torch.zeros_like(log_mu), torch.zeros_like(log_nu)
    for _ in range(iters):
        u = log_mu - torch.logsumexp(Z + v[:, None, :], 2)
        v = log_nu - torch.logsumexp(Z + u[:, :, None], 1)
    ref = Z + u[:, :, None] + v[:, None, :] - norm
    (ref * w.double()).sum().backward()
    assert (out.detach().double() - ref.detach()).abs().max().item() < 2e-4
    assert rel_err(sim.grad, sd.grad) < 1e-4, rel_err(sim.grad, sd.grad)
    assert abs(alpha.grad.item() - ad.grad.item()) < 1e-4 * max(1.0, abs(ad.grad.item()))
    # the tensor-math statement of the reverse sweep (pinned on the CPU to the reference's autograd) agrees too
    if iters and M * N <= 1000 * 777:
        ds2, da2 = heads_grad.log_optimal_transport_backward(sim.detach(), alpha.detach(), iters, w)
        assert rel_err(sim.grad, ds2) < 1e-4 and abs(alpha.grad.item() - da2.item()) < 1e-3 * max(1.0, abs(da2.item()))


@pytest.mark.parametrize("B,M,N,density", [(2, 2048, 2048, 0.0005), (3, 1000, 784, 0.3), (1, 70, 4096, 1.0),
                                             (2, 150, 203, 0.05)])
def test_mask_counts(B, M, N, density):
    """One-pass row / column counts of the ground-truth mask (lightglue.py:595-600 `gt.sum(2)`, `gt.sum(1)`): exact."""
    mask = (torch.rand(B, M, N, generator=torch.Generator().manual_seed(3)) < density).to(DEV)
    r, c = ops.mask_counts(mask.view(torch.uint8))
    assert torch.equal(r, mask.sum(2).float()) and torch.equal(c, mask.sum(1).float())


@pytest.mark.parametrize("kd", [2, 4])
def test_posenc_theta_weight_gradient(kd):
    T = 2 * 3 * 1111
    kp = _rand(T, kd, seed=8)
    w = (_rand(32, kd, seed=9)).requires_grad_()
    gth = _rand(T, 32, seed=10)
    th = ops.PosencTheta.apply(kp, w)
    (th * gth).sum().backward()
    w64 = w.detach().double().requires_grad_()
    ((kp.double() @ w64.t()) * gth.double()).sum().backward()
    assert rel_err(th, kp.double() @ w64.t()) < 1e-6
    assert rel_err(w.grad, w64.grad) < 1e-5


def test_gt_from_homography_matches_reference_labels():
    """Device GT labels (SURVEY 8f row 1) are bit-exact against the reference function's own output (golden) ..."""
    g = dict(np.load(os.path.join(GOLDEN, "gt_homography.npz")))
    for tag in ["a", "b"]:
        kp0, kp1, H = (torch.from_numpy(g[f"{tag}|{n}"]).to(DEV) for n in ("kp0", "kp1", "H"))
        r = ops.gt_matches_from_homography(kp0, kp1, H, 3.0, 3.0)
        assert np.array_equal(r["matches0"].cpu().numpy(), g[f"{tag}|matches0"])
        assert np.array_equal(r["matches1"].cpu().numpy(), g[f"{tag}|matches1"])
        assert np.array_equal(r["assignment"].nonzero().cpu().numpy(), g[f"{tag}|positives"])
        np.testing.assert_allclose(r["proj_0to1"].cpu().numpy(), g[f"{tag}|proj_0to1"], rtol=1e-5, atol=1e-3)
        # the drop-in ground_truth component (mirror of matchers/homography_matcher.py) returns the same labels
        from gluefactory_b200.matchers.homography_matcher import HomographyMatcher
        pred = HomographyMatcher({"th_positive": 3.0, "th_negative": 3.0})({"keypoints0": kp0, "keypoints1": kp1, "H_0to1": H})
        assert np.array_equal(pred["matches0"].cpu().numpy(), g[f"{tag}|matches0"])
        assert pred["assignment"].dtype == torch.bool and set(pred) >= {"matches1", "matching_scores0", "proj_1to0"}


@pytest.mark.parametrize("B,M,N", [(2, 2048, 2048), (3, 1000, 777), (1, 5, 3000)])
def test_gt_from_homography_matches_restatement_at_size(B, M, N):
    """... and against the torch restatement (same warped points) at the benchmark size and on ragged shapes."""
    from gluefactory_b200 import synthetic

    d = synthetic.to_device(synthetic.make_pairs(B, N, seed=70 + B, M=M, with_gt=False), DEV)
    kp0, kp1, H = d["keypoints0"], d["keypoints1"], d["H_0to1"]
    asg, m0, m1 = synthetic.gt_matches_from_homography(kp0, kp1, H, 3.0, 3.0)
    r = ops.gt_matches_from_homography(kp0, kp1, H, 3.0, 3.0)
    assert torch.equal(r["matches0"], m0) and torch.equal(r["matches1"], m1)
    assert torch.equal(r["assignment"], asg)
    assert int(asg.sum()) > 0
    sparse = ops.gt_matches_from_homography(kp0, kp1, H, 3.0, 3.0, dense=False, dense_t=True)
    assert "assignment" not in sparse and torch.equal(sparse["matches0"], m0)
    assert torch.equal(sparse["assignment_t"], asg.transpose(1, 2))  # the transposed mask written in the same pass


def test_gt_from_pose_depth_matches_reference_labels():
    """SURVEY 8f row 1, second half: labels of gt_matches_from_pose_depth (geometry/gt_generation.py:13-106) -- th_epi
    None / 5, th_consistency None / 3 -- bit-exact against the reference function's own output (golden), (a) for the
    O(M N) kernels alone on the reference's reprojections and masks, (b) through the drop-in depth_matcher component
    with duck-typed Camera / Pose objects."""
    from gluefactory_b200 import synthetic
    from gluefactory_b200.matchers.depth_matcher import DepthMatcher

    g = dict(np.load(os.path.join(GOLDEN, "gt_pose_depth.npz")))
    for tag in "abc":
        B, M, N, seed, epi, cc = g[f"{tag}|meta"]
        B, M, N, seed = int(B), int(M), int(N), int(seed)
        sc = synthetic.to_device(synthetic.pose_depth_scene(B, M, N, seed), DEV)
        conf = {"th_positive": 3.0, "th_negative": 5.0, "th_epi": None if epi < 0 else float(epi),
                "th_consistency": None if cc < 0 else float(cc)}
        data = {"keypoints0": sc["kp0"], "keypoints1": sc["kp1"],
                "view0": {"camera": synthetic.PinholeCamera(sc["K0"]), "depth": sc["depth0"]},
                "view1": {"camera": synthetic.PinholeCamera(sc["K1"]), "depth": sc["depth1"]},
                "T_0to1": synthetic.RigidPose(sc["R"], sc["t"])}
        pred = DepthMatcher(conf)(data)
        assert np.array_equal(pred["matches0"].cpu().numpy(), g[f"{tag}|matches0"]), tag
        assert np.array_equal(pred["matches1"].cpu().numpy(), g[f"{tag}|matches1"]), tag
        assert np.array_equal(pred["assignment"].nonzero().cpu().numpy(), g[f"{tag}|positives"]), tag
        assert np.array_equal(pred["visible0"].cpu().numpy(), g[f"{tag}|visible0"])
        if epi < 0:  # kernel alone, from the reference's own reprojections / masks
            t = lambda k: torch.from_numpy(g[f"{tag}|{k}"]).to(DEV)  # noqa: E731
            r = ops.gt_matches_from_reprojection(sc["kp0"], sc["kp1"], t("proj_0to1"), t("proj_1to0"), t("visible0"),
                                                 t("visible1"), t("valid0"), t("valid1"), 3.0, 5.0)
            assert np.array_equal(r["matches0"].cpu().numpy(), g[f"{tag}|matches0"])
            assert np.array_equal(r["matches1"].cpu().numpy(), g[f"{tag}|matches1"])
    torch.cuda.synchronize()


def test_gt_from_homography_degenerate_rows():
    """Rows / columns whose distances are all +inf or NaN (overflowing or NaN keypoints, a point on the homography's
    line at infinity) must behave like torch's min (valid first index, NaN propagates), never index out of bounds."""
    from gluefactory_b200 import synthetic

    d = synthetic.to_device(synthetic.make_pairs(2, 300, seed=91, M=260, with_gt=False), DEV)
    kp0, kp1, H = d["keypoints0"].clone(), d["keypoints1"].clone(), d["H_0to1"]
    kp0[0, 7] = 3e30                      # squared distances overflow to +inf for the whole row
    kp1[0, 11] = float("nan")             # a NaN column
    kp1[1, 5] = float("inf")
    kp0[1, 0] = float("nan")
    asg, m0, m1 = synthetic.gt_matches_from_homography(kp0, kp1, H, 3.0, 3.0)
    r = ops.gt_matches_from_homography(kp0, kp1, H, 3.0, 3.0)
    torch.cuda.synchronize()
    assert torch.equal(r["matches0"], m0) and torch.equal(r["matches1"], m1)
    assert torch.equal(r["assignment"], asg)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 2e-5), (torch.bfloat16, 1.5e-2)])
def test_gluestick_attention_matches_golden(dtype, tol):
    """SURVEY 8a row a15: GlueStick's channels-first attention core (gluestick.py:524-529), forward and gradients,
    against vectors produced by the reference function itself (oracle/make_golden.py)."""
    g = load_gluestick_attn()
    q, k, v = (torch.from_numpy(g[f"core|{n}"]).to(dtype).to(DEV).requires_grad_() for n in "qkv")
    out = ops.gluestick_attention(q, k, v)
    assert out.shape == q.shape
    if dtype == torch.float32:
        assert rel_err(out, torch.from_numpy(g["core|out"])) < tol
        (out * torch.from_numpy(g["core|w"]).float().to(DEV)).sum().backward()
        for n, t in (("dq", q), ("dk", k), ("dv", v)):
            assert rel_err(t.grad, torch.from_numpy(g[f"core|{n}"])) < tol, n
    else:  # bf16 operands: compare with the oracle evaluated on the same rounded operands
        from oracle import lightglue_oracle as O
        qd, kd, vd = (t.detach().double().cpu().requires_grad_() for t in (q, k, v))
        ref = O.gluestick_attention(qd, kd, vd)
        assert rel_err(out, ref) < tol
        w = torch.from_numpy(g["core|w"])
        (ref * w).sum().backward()
        (out.float() * w.float().to(DEV)).sum().backward()
        for n, t, td in (("dq", q, qd), ("dk", k, kd), ("dv", v, vd)):
            assert rel_err(t.grad, td.grad) < 3e-2, n


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("rows,cols", [(16384, 256), (1000, 768), (37, 8), (4096, 512)])
def test_colsum_and_residual(dtype, rows, cols):
    a = _rand(rows, cols, seed=1, dtype=dtype)
    ref = a.double().sum(0)
    assert rel_err(ops.colsum(a), ref) < 1e-5
    x = _rand(rows, cols, seed=2)
    xo, xc = ops.residual_add_cast(x, a, dtype)
    assert torch.equal(xo, x + a.float())
    assert torch.equal(xc, (x + a.float()).to(dtype))
    _, xc2 = ops.residual_add_cast(x, None, dtype)
    assert torch.equal(xc2, x.to(dtype))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("T,D,has_tok", [(4096, 256, True), (1001, 128, False), (777, 512, True), (5, 64, True)])
def test_head_token_kernels(dtype, T, D, has_tok):
    """Fused matchability / token-confidence heads (lightglue.py:74-83, 259-267) against torch in fp64."""
    x = _rand(T, D, seed=1)
    wm, bm = _rand(1, D, seed=2) * 0.1, _rand(1, seed=3)
    wt, bt = (_rand(1, D, seed=4) * 0.1, _rand(1, seed=5)) if has_tok else (None, None)
    xc, zt, ls, du = ops.head_token_fwd(x, wm.view(-1), bm, wt.view(-1) if has_tok else None, bt, dtype)
    assert torch.equal(xc, x.to(dtype))
    z0 = x.double() @ wm.double().t() + bm.double()
    z1 = x.double() @ wt.double().t() + bt.double() if has_tok else z0
    assert rel_err(zt, torch.cat([z0, z1], 1)) < 1e-5
    assert rel_err(ls, torch.nn.functional.logsigmoid(z0[:, 0])) < 1e-5
    assert rel_err(du, torch.nn.functional.logsigmoid(-z0[:, 0])) < 1e-5
    # backward
    dmdw = _rand(T, D, seed=6, dtype=dtype)
    dzt = _rand(T, 2, seed=7)
    for _ in range(2):  # second call checks the self-resetting arrival counter
        dx, dW2, db2 = ops.head_token_bwd(x, dmdw, dzt, wm.view(-1))
        assert rel_err(dx, dmdw.double() + dzt[:, :1].double() * wm.double()) < 1e-6
        assert rel_err(dW2, dzt.double().t() @ x.double()) < 1e-5
        assert rel_err(db2, dzt.double().sum(0)) < 1e-5


def test_adam_flat_matches_torch():
    n = 100_003
    p = _rand(n, seed=1)
    ref = torch.nn.Parameter(p.clone())
    opt = torch.optim.Adam([ref], lr=1e-3, weight_decay=0.01)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    for t in range(1, 4):
        g = _rand(n, seed=10 + t)
        ref.grad = g.clone()
        opt.step()
        ops.adam_flat_(p, g * 4.0, m, v, t, 1e-3, weight_decay=0.01, grad_scale=0.25)
    assert rel_err(p, ref.data) < 1e-6


def test_errors_are_reported():
    from gluefactory_b200._lib import Lgb200Error, call, stream_ptr

    with pytest.raises(Lgb200Error, match="null pointer"):
        call("lgb200_assign_lse", None, None, None, None, 1, 4, 4, stream_ptr())
    with pytest.raises(Lgb200Error, match="empty"):
        x = torch.zeros(4, device=DEV)
        from gluefactory_b200._lib import ptr
        call("lgb200_assign_lse", ptr(x), ptr(x), ptr(x), ptr(x), 0, 4, 4, stream_ptr())
