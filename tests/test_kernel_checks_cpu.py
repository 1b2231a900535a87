"""The comparison helpers of tests/kernel_checks.py must see the defects a global relative L2 error hides.

Each case takes an fp64 reference and an honest result (fp32 arithmetic rounded to bf16 exactly where the kernels round),
checks that the honest result passes, then injects one defect and checks that the per-element bound or the per-block
check rejects it, while the old global rel-L2 < 1e-2 check still accepts it.  No GPU needed."""
import math

import pytest
import torch

from kernel_checks import (assert_gaps_untouched, attention_bwd_ref_bound, attention_fwd_ref_bound, canary_view, ce_ref_bound,
                           check_blocks, check_bounded, gemm_ref_bound, global_rel_l2, layernorm_bwd_ref_bound,
                           layernorm_fwd_ref_bound)

OLD_BAR = 1e-2


def _fails(fn, *a, **kw):
    try:
        fn(*a, **kw)
    except AssertionError as e:
        return str(e)
    return None


@pytest.fixture(scope="module")
def gemm_case():
    g = torch.Generator().manual_seed(0)
    M, N, K = 14592, 512, 768
    a = (torch.randn(M, K, generator=g) * 0.5).to(torch.bfloat16)
    b = (torch.randn(N, K, generator=g) * 0.5).to(torch.bfloat16)
    ref, bound, _ = gemm_ref_bound(a, b)
    honest = (a.float() @ b.float().t()).to(torch.bfloat16)
    return ref, bound, honest


def test_gemm_honest_passes(gemm_case):
    ref, bound, honest = gemm_case
    worst = check_bounded("gemm", honest, ref, bound)
    print("honest gemm: max err/bound %.3f" % worst)
    check_blocks(honest, ref, (128, ref.shape[1]), 1e-2)


def test_gemm_last_row_zeroed_is_caught(gemm_case):
    ref, bound, honest = gemm_case
    bad = honest.clone()
    bad[-1] = 0
    assert global_rel_l2(bad, ref) < OLD_BAR
    assert _fails(check_bounded, "gemm", bad, ref, bound)
    assert _fails(check_blocks, bad, ref, (1, ref.shape[1]), 1e-2)


def test_gemm_last_tile_scaled_is_caught(gemm_case):
    ref, bound, honest = gemm_case
    bad = honest.clone()
    bad[-128:] = (bad[-128:].float() * 1.05).to(torch.bfloat16)
    assert global_rel_l2(bad, ref) < OLD_BAR
    assert _fails(check_bounded, "gemm", bad, ref, bound)
    assert _fails(check_blocks, bad, ref, (128, ref.shape[1]), 1e-2)


def _honest_attention(q, k, v, B, heads, S, add):
    """fp32 scores and softmax numerators, P rounded to bf16 for P.V, fp32 row sum, bf16 output - the kernels' rounding"""
    W = q.shape[1]
    d = W // heads
    sh = lambda t: t.float().view(B, S, heads, d).transpose(1, 2)
    s2 = (sh(q) @ sh(k).transpose(-1, -2)) * (1.4426950408889634 / math.sqrt(d)) + add.view(B, 1, 1, S) * 1.4426950408889634
    p = torch.exp2(s2 - s2.amax(-1, keepdim=True))
    o = (p.to(torch.bfloat16).float() @ sh(v)) / p.sum(-1, keepdim=True)
    return o.transpose(1, 2).reshape(B * S, W).to(torch.bfloat16)


@pytest.fixture(scope="module")
def attn_case():
    g = torch.Generator().manual_seed(1)
    B, heads, S, d = 40, 12, 228, 64
    W = heads * d
    q, k, v = ((torch.randn(B * S, W, generator=g) * 0.8).to(torch.bfloat16) for _ in range(3))
    lens = torch.randint(S // 2, S + 1, (B,), generator=g)
    add = ((torch.arange(S)[None, :] >= lens[:, None]).float() * -10000.0)
    ctx, bound, _, _ = attention_fwd_ref_bound(q, k, v, B, heads, S, S, mask=add)
    honest = _honest_attention(q, k, v, B, heads, S, add)
    return dict(B=B, heads=heads, S=S, d=d, q=q, k=k, v=v, add=add, lens=lens, ctx=ctx, bound=bound, honest=honest)


def _head_blocks(c):
    # [B*S, W] viewed as [B, S, heads, d]: one block per (sample, head)
    return lambda t: t.view(c["B"], c["S"], c["heads"], c["d"]), (1, c["S"], 1, c["d"])


def test_attention_honest_passes(attn_case):
    c = attn_case
    worst = check_bounded("ctx", c["honest"], c["ctx"], c["bound"])
    view, blk = _head_blocks(c)
    wb = check_blocks(view(c["honest"]), view(c["ctx"]), blk, 1e-2)
    print("honest attention: max err/bound %.3f, worst (sample, head) rel-L2 %.2e" % (worst, wb))


def test_attention_last_head_scaled_is_caught(attn_case):
    c = attn_case
    view, blk = _head_blocks(c)
    bad = view(c["honest"]).clone()
    bad[:, :, -1] = (bad[:, :, -1].float() * 1.02).to(torch.bfloat16)
    assert global_rel_l2(bad, view(c["ctx"])) < OLD_BAR
    assert _fails(check_blocks, bad, view(c["ctx"]), blk, 1e-2)


def test_attention_dropped_key_is_caught(attn_case):
    c = attn_case
    add = c["add"].clone()
    # the last live key of the longest sample is lost: the key with the least weight, so the smallest global trace (a
    # key of a short sample moves the global error to 1.2e-2 .. 1.6e-2 with this data, right at the old bar)
    b = int(c["lens"].argmax())
    add[b, int(c["lens"][b]) - 1] = -10000.0
    bad = _honest_attention(c["q"], c["k"], c["v"], c["B"], c["heads"], c["S"], add)
    view, blk = _head_blocks(c)
    print("dropped key: global rel-L2 %.2e" % global_rel_l2(bad, c["ctx"]))
    assert global_rel_l2(bad, c["ctx"]) < OLD_BAR
    assert _fails(check_blocks, view(bad), view(c["ctx"]), blk, 1e-2)
    assert _fails(check_bounded, "ctx", bad, c["ctx"], c["bound"])


def test_attention_backward_bounds_hold_for_honest_fp32():
    g = torch.Generator().manual_seed(2)
    B, heads, S, d = 3, 2, 100, 64
    W = heads * d
    q, k, v, do = ((torch.randn(B * S, W, generator=g) * 0.8).to(torch.bfloat16) for _ in range(4))
    add = torch.zeros(B, S)
    add[1, 60:] = -10000.0
    dq, dk, dv, bdq, bdk, bdv = attention_bwd_ref_bound(q, k, v, do, B, heads, S, S, mask=add)
    qf, kf, vf = (t.float().view(B, S, W).requires_grad_(True) for t in (q, k, v))
    from oracle import fusion_oracle as O
    out, _ = O.attention_core(qf, kf, vf, add[:, None, None, :], heads)
    out.backward(do.float().view(B, S, W))
    for name, got, ref, bnd in (("dq", qf.grad, dq, bdq), ("dk", kf.grad, dk, bdk), ("dv", vf.grad, dv, bdv)):
        check_bounded(name, got.reshape(B * S, W).to(torch.bfloat16), ref, bnd)
    # a key whose gradient is dropped is seen per element
    bad = vf.grad.reshape(B * S, W).clone()
    bad[S + 5] = 0
    assert _fails(check_bounded, "dv", bad, dv, bdv)


def test_layernorm_bounds_hold_for_honest_fp32():
    g = torch.Generator().manual_seed(3)
    M, H = 257, 1032
    y = torch.randn(M, H, generator=g).to(torch.bfloat16)
    y[5] = 0.75                                          # constant row: var = 0
    gamma = (1 + 0.1 * torch.randn(H, generator=g)).to(torch.bfloat16)
    beta = (0.1 * torch.randn(H, generator=g)).to(torch.bfloat16)
    x, mean, rstd, bx, bm, br = layernorm_fwd_ref_bound(y, gamma, beta)
    yf = y.float().requires_grad_(True)
    out = torch.nn.functional.layer_norm(yf, (H,), gamma.float(), beta.float(), 1e-12)
    check_bounded("x", out.to(torch.bfloat16), x, bx)
    assert torch.equal(x[5], beta.double())
    check_bounded("mean", yf.detach().mean(1), mean, bm)
    dx = torch.randn(M, H, generator=g).to(torch.bfloat16)
    out.backward(dx.float())
    dy, dz, bdy, bdz, dgam, bdg, dbet, bdb, dbias, bdbias = layernorm_bwd_ref_bound(dx, y, gamma)
    rows = torch.arange(M) != 5       # torch's CPU variance of the constant row is not exactly 0, the kernels' is
    check_bounded("dy", yf.grad.to(torch.bfloat16)[rows], dy[rows], bdy[rows])
    xh = (y.float() - y.float().mean(1, keepdim=True)) * torch.rsqrt(y.float().var(1, unbiased=False, keepdim=True) + 1e-12)
    xh[5] = 0
    check_bounded("dgamma", (dx.float() * xh).sum(0), dgam, bdg)
    check_bounded("dbeta", dx.float().sum(0), dbet, bdb)
    bad = (dx.float() * xh).sum(0)
    print("dgamma bound / |dgamma|: median %.2e" % (bdg / dgam.abs()).median().item())
    bad[-1] += 0.05 * dgam.abs().mean().item()
    assert _fails(check_bounded, "dgamma", bad, dgam, bdg)


def test_cross_entropy_bounds_hold_for_honest_fp32():
    g = torch.Generator().manual_seed(4)
    M, V = 64, 30528
    z = (torch.randn(M, V, generator=g) * 3).to(torch.bfloat16)
    labels = torch.randint(0, V, (M,), generator=g)
    labels[0], labels[1], labels[2], labels[3] = 0, V - 1, V - 3, -1
    loss, bl, d, bd = ce_ref_bound(z, labels, 0.25)
    zf = z.float()
    lf = torch.nn.functional.cross_entropy(zf, labels, ignore_index=-1, reduction="none")
    check_bounded("row_loss", lf, loss, bl)
    df = (torch.softmax(zf, 1) - torch.nn.functional.one_hot(labels.clamp_min(0), V).float()) * 0.25
    df[3] = 0
    check_bounded("dlogits", df.to(torch.bfloat16), d, bd)
    bad = lf.clone()
    bad[1] += 1e-2
    assert _fails(check_bounded, "row_loss", bad, loss, bl)


def test_canary_sees_a_write_one_past_the_view():
    view, base = canary_view((37, 24), torch.bfloat16, pad_rows=4, pad_cols=8, device="cpu")
    view.fill_(1.0)
    assert_gaps_untouched(base, view)
    base[2, 24] = 0                      # first row of the view (it starts 2 rows in), one element past its end
    assert _fails(assert_gaps_untouched, base, view)
    view, base = canary_view((5, 8), torch.float32, pad_rows=2, pad_cols=4, device="cpu")
    view.fill_(0.0)
    base[6, 0] = 0                       # one row past the end
    assert _fails(assert_gaps_untouched, base, view)


def test_nan_read_past_the_view_turns_the_output_non_finite():
    a, abase = canary_view((16, 40), torch.bfloat16, pad_rows=2, pad_cols=8, fill=float("nan"), device="cpu")
    a.copy_(torch.randn(16, 40).to(torch.bfloat16))
    b = torch.randn(24, 40).to(torch.bfloat16)
    ref, bound, _ = gemm_ref_bound(a, b)
    good = (a.float() @ b.float().t()).to(torch.bfloat16)
    check_bounded("c", good, ref, bound)
    wide = abase[1:17, :41]              # a kernel that reads one column too many
    bad = (wide.float()[:, :40] @ b.float().t() + wide.float()[:, 40:] * 0).to(torch.bfloat16)
    msg = _fails(check_bounded, "c", bad, ref, bound)
    assert msg and "non-finite" in msg
