"""The CUDA kernels element by element against fp64, at tail shapes, with exact probes and out-of-bounds canaries.

Every comparison is per element against a bound derived in tests/kernel_checks.py (or exact, for the probes whose
result is representable), plus per-block relative L2 where a block-wide scale error could hide under the per-element
bound.  Inputs live in NaN-padded buffers, so a read outside them turns an output non-finite; outputs live inside
sentinel buffers whose gaps must come back bit for bit.  Each case prints max(err / bound)."""
import math

import pytest
import torch

from kernel_checks import (U16, U32, assert_gaps_untouched, attention_bwd_ref_bound, attention_fwd_ref_bound, canary_view,
                           ce_ref_bound, check_blocks, check_bounded, epi_bound_gelu, epi_bound_gelu_bwd, gemm_ref_bound,
                           layernorm_bwd_ref_bound, layernorm_fwd_ref_bound)

pytestmark = pytest.mark.gpu

NAN = float("nan")


def _F():
    from mmf_b200 import functional as F, lib
    return F, lib


def _nan_input(t, pad_rows=2, pad_cols=16):
    """t copied into a NaN-padded buffer (gap rows before and after, pad_cols NaN columns after each row)"""
    view, base = canary_view(tuple(t.shape), t.dtype, pad_rows, pad_cols, fill=NAN)
    view.copy_(t)
    return view, base


def _report(tag, **ratios):
    print("%s: %s" % (tag, " ".join("%s=%.3f" % kv for kv in ratios.items())))


# ======================================================================================================================
# GEMM
# ======================================================================================================================
LAYOUTS = [(False, False), (False, True), (True, False), (True, True)]
M_CLASSES = [1, 8, 129, 264, 1160, 14600]
N_CLASSES = [8, 136, 264, 776, 2312, 30528]
K_CLASSES = [8, 40, 72, 1000, 3080]


def _onehot_cases():
    """About 30 combinations: every M, N and K class meets every layout (an MN-major A needs M % 8 == 0, so M = 1 and 129
    meet the K-major-A layouts only), with block_n 128 / 256 and cluster 1 / 2 alternating; large M pairs with small N so
    the whole set stays fast."""
    cases = []
    i = 0
    for li, (a_mn, b_mn) in enumerate(LAYOUTS):
        ms = [m for m in M_CLASSES if not (a_mn and m % 8)]
        for j in range(6):
            M = ms[(j + li) % len(ms)]
            N = N_CLASSES[(j + 2 * li) % 6]
            K = K_CLASSES[(j + li) % 5]
            if M * N > 60_000_000:
                N = 776
            cases.append((a_mn, b_mn, M, N, K, 128 if i % 2 else 256, 1 + (i // 2) % 2))
            i += 1
    for j, K in enumerate(K_CLASSES):       # every K class once more where N has a 128-tile tail and M a 128-row tail
        cases.append((j % 2 == 0, j % 2 == 0, 264, 136 + 128 * j, K, 256 if j % 2 else 128, 2 - j % 2))
    for li, (a_mn, b_mn) in enumerate(LAYOUTS):
        # the vocabulary width where the cap above took it away, with the smallest M that still makes a CTA pair
        if not any(c[:2] == (a_mn, b_mn) and c[3] == N_CLASSES[-1] for c in cases):
            cases.append((a_mn, b_mn, 264 if a_mn else 129, N_CLASSES[-1], K_CLASSES[li + 1], 256, 2))
    return cases


def _perm(M, K):
    return (7919 * torch.arange(M, device="cuda", dtype=torch.int64)) % K


def _onehot_a(M, K):
    a = torch.zeros(M, K, dtype=torch.bfloat16, device="cuda")
    a[torch.arange(M, device="cuda"), _perm(M, K)] = 1.0
    return a


def _store(t, mn):
    """logical [rows, K] operand -> (stored operand as a column slice of a NaN-padded buffer, base)"""
    st = t.t().contiguous() if mn else t
    return _nan_input(st)


@pytest.mark.parametrize("a_mn,b_mn,M,N,K,bn,cluster", _onehot_cases())
def test_gemm_onehot_probe_exact(a_mn, b_mn, M, N, K, bn, cluster):
    """A[i, (7919 i) mod K] = 1 selects one column of B per output row, so C[i, j] = B[j, pi(i)] exactly: a misplaced tile,
    row, column or k-block, or a stale accumulator, changes some element.  No tolerance."""
    F, lib = _F()
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    a = _onehot_a(M, K)
    b = torch.randn(N, K, generator=g, device="cuda").to(torch.bfloat16)
    a_st, _ = _store(a, a_mn)
    b_st, _ = _store(b, b_mn)
    want = b[:, _perm(M, K)].t()
    out, obase = canary_view((M, N), torch.bfloat16, 4, 8)
    c = F.gemm(a_st, b_st, a_mn=a_mn, b_mn=b_mn, epi=lib.EPI_BIAS, out=out, block_n=bn, cluster=cluster)
    torch.cuda.synchronize()
    assert c.data_ptr() == out.data_ptr()
    assert torch.equal(c, want), "max |diff| %.3g" % (c.float() - want.float()).abs().max().item()
    assert_gaps_untouched(obase, out, name="C")
    if a_mn and b_mn:
        # the fp32 wgrad epilogue (red.global into a zeroed view of a sentinel buffer), over split-K counts that leave
        # one k-block per split, uneven splits and more splits than k-blocks
        kb = (K + 63) // 64
        for splits in sorted({1, 3, 7, kb + 5}):
            o32, b32 = canary_view((M, N), torch.float32, 2, 4)
            o32.zero_()
            F.gemm(a_st, b_st, a_mn=True, b_mn=True, epi=lib.EPI_ATOMIC_F32, out=o32, splits=splits, block_n=bn,
                   cluster=cluster)
            torch.cuda.synchronize()
            assert torch.equal(o32, want.float()), "splits=%d" % splits
            assert_gaps_untouched(b32, o32, name="C32")
    print("onehot a_mn=%d b_mn=%d %dx%dx%d bn=%d cluster=%d: exact" % (a_mn, b_mn, M, N, K, bn, cluster))


def _rand(rows, cols, g, scale=0.5):
    return (torch.randn(rows, cols, generator=g, device="cuda") * scale).to(torch.bfloat16)


@pytest.mark.parametrize("M,N,K,cluster", [(200, 776, 72, 2), (200, 776, 1000, 1), (1160, 264, 1032, 2), (129, 136, 40, 1)])
def test_gemm_epilogues_per_element(M, N, K, cluster):
    """Every epilogue on random data where M and N both have tails, against fp64 with the derived bound.  Operands, aux
    and the keep-bit words are column slices of NaN-padded buffers; outputs are views in sentinel buffers."""
    F, lib = _F()
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    a, w = _rand(M, K, g), _rand(N, K, g)
    a_st, _ = _nan_input(a)
    w_st, _ = _nan_input(w)
    bias = (torch.randn(N, generator=g, device="cuda") * 0.5).to(torch.bfloat16)
    ref, bnd, accb = gemm_ref_bound(a, w, bias)
    r = {}
    # bias
    out, ob = canary_view((M, N), torch.bfloat16, 2, 8)
    F.gemm(a_st, w_st, epi=lib.EPI_BIAS, bias=bias, out=out, cluster=cluster)
    r["bias"] = check_bounded("bias", out, ref, bnd)
    assert_gaps_untouched(ob, out)
    # bias + relu
    out, ob = canary_view((M, N), torch.bfloat16, 2, 8)
    F.gemm(a_st, w_st, epi=lib.EPI_BIAS_RELU, bias=bias, out=out, cluster=cluster)
    r["relu"] = check_bounded("relu", out, ref.clamp_min(0), bnd)
    assert_gaps_untouched(ob, out)
    # bias + gelu: u and h through one ldc
    ub, ubase = canary_view((M, N), torch.bfloat16, 2, 8)
    hb, hbase = canary_view((M, N), torch.bfloat16, 2, 8)
    F.gemm(a_st, w_st, epi=lib.EPI_BIAS_GELU, bias=bias, out=ub, out2=hb, cluster=cluster)
    r["gelu_u"] = check_bounded("gelu u", ub, ref, bnd)
    h_ref, h_bnd = epi_bound_gelu(ref, accb)
    r["gelu_h"] = check_bounded("gelu h", hb, h_ref, h_bnd)
    assert_gaps_untouched(ubase, ub, name="u")
    assert_gaps_untouched(hbase, hb, name="h")
    # a strided u with the default h: the wrapper allocates h with u's row stride, which the kernel writes it with
    ub, ubase = canary_view((M, N), torch.bfloat16, 2, 8)
    u2, h2 = F.gemm(a_st, w_st, epi=lib.EPI_BIAS_GELU, bias=bias, out=ub, cluster=cluster)
    assert u2.data_ptr() == ub.data_ptr() and h2.stride(0) == ub.stride(0)
    r["gelu_h_default"] = check_bounded("gelu h (default out2)", h2, h_ref, h_bnd)
    assert_gaps_untouched(ubase, ub, name="u")
    # bias + dropout (N % 32 != 0: a partial last keep word) + residual
    keep = torch.rand(M, N, generator=g, device="cuda") >= 0.1
    words, _ = _nan_input(F.pack_keep_bits(keep).view(torch.float32), pad_cols=4)
    words = words.view(torch.int32)
    resid = _rand(M, N, g, 1.0)
    resid_st, _ = _nan_input(resid)
    scale = 1 / 0.9
    kd = keep.double() * scale
    y_ref = ref * kd + resid.double()
    # (acc + bias) * keep * scale + resid in fp32: the accumulator error scaled, one rounding each for the scale and the add
    y_bnd = U16 * y_ref.abs() + (1 + U16) * (accb * kd + U32 * (ref * kd).abs() + U32 * y_ref.abs())
    for cl in (1, 2):
        out, ob = canary_view((M, N), torch.bfloat16, 2, 8)
        F.gemm(a_st, w_st, epi=lib.EPI_BIAS_DROP_RESID, bias=bias, aux=resid_st, drop_mask=words, drop_scale=scale, out=out,
               cluster=cl)
        r["drop_resid_c%d" % cl] = check_bounded("drop+resid cluster %d" % cl, out, y_ref, y_bnd)
        assert_gaps_untouched(ob, out)
    # dgrad epilogues: B MN-major, aux = pre-activation, strided
    dy = _rand(M, N, g)
    dy_st, _ = _nan_input(dy)
    wk = _rand(N, K, g, 0.05)                      # [out = N, in = K]: dX = dY W, B[n=K, k=N] stored [N, K] = MN-major
    wk_st, _ = _nan_input(wk)
    pre = _rand(M, K, g, 1.0)
    pre_st, _ = _nan_input(pre)
    dref, dbnd, daccb = gemm_ref_bound(dy, wk.t().contiguous())
    out, ob = canary_view((M, K), torch.bfloat16, 2, 8)
    F.gemm(dy_st, wk_st, b_mn=True, epi=lib.EPI_GELU_BWD, aux=pre_st, out=out, cluster=cluster)
    gref, gbnd = epi_bound_gelu_bwd(dref, daccb, pre)
    r["gelu_bwd"] = check_bounded("gelu_bwd", out, gref, gbnd)
    assert_gaps_untouched(ob, out)
    out, ob = canary_view((M, K), torch.bfloat16, 2, 8)
    F.gemm(dy_st, wk_st, b_mn=True, epi=lib.EPI_ADD_AUX, aux=pre_st, out=out, cluster=cluster)
    aref = dref + pre.double()
    r["add_aux"] = check_bounded("add_aux", out, aref, U16 * aref.abs() + (1 + U16) * (daccb + U32 * aref.abs()))
    assert_gaps_untouched(ob, out)
    # wgrad: dW[N, K] += dY^T X, split-K, twice (accumulates)
    if M % 8 == 0:
        x = _rand(M, K, g)
        x_st, _ = _nan_input(x)
        wref, wbnd, _ = gemm_ref_bound(dy.t().contiguous(), x.t().contiguous(), out_bf16=False)
        for splits in (1, 3):
            o32, b32 = canary_view((N, K), torch.float32, 2, 4)
            o32.zero_()
            F.gemm(dy_st, x_st, a_mn=True, b_mn=True, epi=lib.EPI_ATOMIC_F32, out=o32, splits=splits, cluster=cluster)
            F.gemm(dy_st, x_st, a_mn=True, b_mn=True, epi=lib.EPI_ATOMIC_F32, out=o32, splits=splits, cluster=cluster)
            r["wgrad_s%d" % splits] = check_bounded("wgrad", o32, 2 * wref, 2 * wbnd + 2 * U32 * wref.abs())
            assert_gaps_untouched(b32, o32)
    torch.cuda.synchronize()
    _report("gemm epilogues %dx%dx%d cluster %d" % (M, N, K, cluster), **r)


def test_gemm_rejects_misshaped_buffers():
    """out / out2 / bias / aux / drop_mask are handed over as pointers: each mis-shaped one is a view inside a larger
    allocation (so a wrapper without the check writes or reads memory it owns) and must raise ValueError."""
    F, lib = _F()
    M, N, K = 64, 256, 64
    a = torch.zeros(M, K, dtype=torch.bfloat16, device="cuda")
    w = torch.zeros(N, K, dtype=torch.bfloat16, device="cuda")
    big = torch.zeros(M + 8, N + 64, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(ValueError):
        F.gemm(a, w, out=big[:M, :N - 8])
    with pytest.raises(ValueError):
        F.gemm(a, w, out=big[:M - 1, :N])
    with pytest.raises(ValueError):
        F.gemm(a, w, epi=lib.EPI_BIAS_GELU, bias=big[0, :N], out2=big[:M, :N - 8])
    with pytest.raises(ValueError):
        F.gemm(a, w, bias=big[0, :N - 8])
    with pytest.raises(ValueError):
        F.gemm(a, w, epi=lib.EPI_BIAS_DROP_RESID, bias=big[0, :N], aux=big[:M - 1, :N])
    words = torch.zeros(M + 8, N // 32 + 4, dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError):
        F.gemm(a, w, epi=lib.EPI_BIAS_DROP_RESID, bias=big[0, :N], aux=big[:M, :N], drop_mask=words[:M, :N // 32 - 1])
    f32 = torch.zeros(N + 8, K + 8, dtype=torch.float32, device="cuda")
    with pytest.raises(ValueError):
        F.gemm(a, a, a_mn=True, b_mn=True, epi=lib.EPI_ATOMIC_F32, out=f32[:K - 1, :K])
    torch.cuda.synchronize()


# ======================================================================================================================
# attention
# ======================================================================================================================
def _mask_patterns(Skv, Sq_hint=0):
    """[B, Skv] 0/1 key masks: none, prefix, suffix (first keys masked), holes (live [0, t) + [T, T + r): text + image),
    single live keys at 0, 31, 32, 127, 128, 255, 256, Skv - 1 and inside the partial last 32-key chunk, one fully masked
    sample.  Returns (mask01, names)."""
    rows, names = [], []
    ar = torch.arange(Skv, device="cuda")

    def add(m, name):
        rows.append(m.long())
        names.append(name)
    add(torch.ones(Skv, device="cuda"), "none")
    add(ar < max(1, (2 * Skv) // 3), "prefix")
    add(ar >= Skv // 3, "suffix")
    t, T = max(1, Skv // 4), max(2, Skv // 2)
    add((ar < t) | ((ar >= T) & (ar < T + max(1, Skv // 5))), "holes")
    for j in sorted({0, 31, 32, 127, 128, 255, 256, Skv - 1, (Skv // 32) * 32 + (Skv % 32) // 2}):
        if j < Skv:
            add(ar == j, "single@%d" % j)
    add(torch.zeros(Skv, device="cuda"), "all-masked")
    return torch.stack(rows), names


def _bf16_ulp(x):
    e = torch.floor(torch.log2(x.abs().clamp_min(1e-30)))
    return torch.where(x == 0, torch.zeros_like(x), torch.exp2(e - 7))


def _uniform_probe(F, B, heads, Sq, Skv, d, mask01, p_drop, g):
    W = heads * d
    q = torch.zeros(B * Sq, W, dtype=torch.bfloat16, device="cuda")
    # v in multiples of 1/64 within [-2, 2]: any sum of up to 384 of them is exact in fp32
    v = (torch.randint(-128, 129, (B * Skv, W), generator=g, device="cuda").float() / 64).to(torch.bfloat16)
    sent = torch.where(torch.rand(B * Skv, W, generator=g, device="cuda") < 0.5, -64.0, 64.0).to(torch.bfloat16)
    live = mask01.reshape(B * Skv, 1).bool()
    allm = (mask01.sum(1) == 0).repeat_interleave(Skv)[:, None]
    v = torch.where(live | allm, v, sent)               # masked keys carry +-64 unless the whole sample is masked
    k = _rand(B * Skv, W, g, 1.0)
    add = ((1.0 - mask01.float()) * -10000.0).contiguous()
    keep = dm = None
    scale = 1.0
    if p_drop:
        keep = torch.rand(B, heads, Sq, Skv, generator=g, device="cuda") >= p_drop
        dm, scale = F.pack_keep_bits(keep), 1.0 / (1.0 - p_drop)
    return q, k, v, add, keep, dm, scale


ATTN_PROBE = [(64, Skv, Sq) for Skv, Sq in [(1, 36), (17, 1), (31, 129), (32, 128), (33, 36), (100, 228), (128, 129),
                                             (129, 1), (228, 228), (256, 256), (257, 36), (300, 300), (384, 129)]] + \
             [(128, Skv, Sq) for Skv, Sq in [(1, 1), (33, 129), (128, 36), (129, 256), (228, 228), (256, 128)]]


@pytest.mark.parametrize("d,Skv,Sq", ATTN_PROBE)
@pytest.mark.parametrize("p_drop", [0.0, 0.25])
def test_attention_uniform_probe_exact(d, Skv, Sq, p_drop):
    """q = 0: every live key gets p = exp2(0) = 1, so ctx_i = scale * sum_{live, kept} v_j / n_live (within one bf16 ulp:
    the sum is exact, the division and the bf16 store round once each) and lse2 = log2(n_live).  Masked keys carry
    +-64 in V, so a leaked key is obvious; a fully masked sample averages all Skv rows with lse2 = log2(Skv) - 10000
    log2(e).  The backward then has dk = 0 exactly and dv within its fp64 bound."""
    F, _ = _F()
    g = torch.Generator(device="cuda").manual_seed(Skv * 1000 + Sq + d)
    mask01, names = _mask_patterns(Skv)
    B, heads = mask01.shape[0], 2
    W = heads * d
    q, k, v, add, keep, dm, scale = _uniform_probe(F, B, heads, Sq, Skv, d, mask01, p_drop, g)
    ctx, lse2 = F.attention_fwd(q, k, v, B, heads, Sq, Skv, mask=add, drop_mask=dm, drop_scale=scale)
    torch.cuda.synchronize()
    n_live = mask01.sum(1).double()
    allm = n_live == 0
    eff = torch.where(allm[:, None], torch.ones_like(mask01), mask01).double()       # keys that get p = 1
    n_eff = eff.sum(1)
    v4 = v.double().view(B, Skv, heads, d).permute(0, 2, 1, 3)                       # [B, h, Skv, d]
    if keep is None:
        num = torch.einsum("bk,bhkd->bhd", eff, v4)[:, :, None, :].expand(B, heads, Sq, d)
    else:
        num = torch.einsum("bk,bhqk,bhkd->bhqd", eff, keep.double(), v4) * scale
    want = (num / n_eff[:, None, None, None]).permute(0, 2, 1, 3).reshape(B * Sq, W)
    r = check_bounded("ctx", ctx, want, _bf16_ulp(want))
    lse_want = torch.log2(n_eff)[:, None, None].expand(B, heads, Sq).clone()
    lse_bnd = torch.full_like(lse_want, 1e-6)
    lse_want[allm] -= 10000.0 / math.log(2.0)
    lse_bnd[allm] = 2 * 2.0 ** (math.floor(math.log2(abs(lse_want[allm].max().item()) if allm.any() else 1)) - 23)
    rl = check_bounded("lse2", lse2, lse_want, lse_bnd)
    # backward: q = 0 gives dk = 0 exactly
    dctx = _rand(B * Sq, W, g, 1.0)
    dq, dk, dv = F.attention_bwd(dctx, q, k, v, ctx, lse2, B, heads, Sq, Skv, mask=add, drop_mask=dm, drop_scale=scale)
    torch.cuda.synchronize()
    assert torch.equal(dk, torch.zeros_like(dk)), "dk must be exactly 0 when q = 0"
    rdq, rdk, rdv, bdq, bdk, bdv = attention_bwd_ref_bound(q, k, v, dctx, B, heads, Sq, Skv, mask=add, keep=keep,
                                                           drop_scale=scale, ctx_lo=False)
    rv = check_bounded("dv", dv, rdv, bdv)
    rq = check_bounded("dq", dq, rdq, bdq)
    _report("uniform d%d Skv%d Sq%d p%.2f (%d masks)" % (d, Skv, Sq, p_drop, B), ctx=r, lse2=rl, dv=rv, dq=rq)


def _attn_random(F, B, heads, Sq, Skv, d, g, p_drop=0.0, holes=True, fused=True):
    """q/k/v as column slices of a fused NaN-padded buffer (NaN columns past 3W, NaN rows after the last sample when
    Sq == Skv); key masks mixing prefix, suffix and holes, one fully masked sample."""
    W = heads * d
    if Sq == Skv and fused:
        base = torch.full((B * Sq + 8, 3 * W + 64), NAN, dtype=torch.bfloat16, device="cuda")
        base[:B * Sq, :3 * W] = _rand(B * Sq, 3 * W, g, 0.8)
        q, k, v = base[:B * Sq, :W], base[:B * Sq, W:2 * W], base[:B * Sq, 2 * W:3 * W]
    else:
        q = _nan_input(_rand(B * Sq, W, g, 0.8))[0]
        k = _nan_input(_rand(B * Skv, W, g, 0.8))[0]
        v = _nan_input(_rand(B * Skv, W, g, 0.8))[0]
    ar = torch.arange(Skv, device="cuda")
    lens = torch.randint(max(1, Skv // 3), Skv + 1, (B,), generator=g, device="cuda")
    mask01 = (ar[None] < lens[:, None]).long()
    if holes and B > 2:
        t = torch.randint(1, max(2, Skv // 2), (B,), generator=g, device="cuda")
        mask01[1::3] = ((ar[None] < t[1::3, None]) | (ar[None] >= Skv // 2)).long()
        mask01[2::3] = (ar[None] >= t[2::3, None]).long()
    mask01[0] = 0
    add = ((1.0 - mask01.float()) * -10000.0).contiguous()
    keep = dm = None
    scale = 1.0
    if p_drop:
        keep = torch.rand(B, heads, Sq, Skv, generator=g, device="cuda") >= p_drop
        dm, scale = F.pack_keep_bits(keep), 1.0 / (1.0 - p_drop)
    return q, k, v, add, mask01, keep, dm, scale


ATTN_RANDOM = [
    # (B, heads, Sq, Skv, d, p_drop, env)
    (40, 12, 228, 228, 64, 0.1, {}),                                     # paired fwd + persistent bwd
    (13, 4, 129, 257, 64, 0.0, {}),                                      # general kernels, d = 64
    (6, 4, 300, 300, 64, 0.1, {}),
    (50, 8, 100, 100, 128, 0.1, {}),                                     # d = 128, 400 items
    (4, 8, 36, 256, 128, 0.0, {}),
    (9, 6, 228, 228, 64, 0.1, {"MMFB_ATTN_FWD": "1", "MMFB_ATTN_BWD": "8"}),
    (9, 6, 129, 33, 64, 0.0, {"MMFB_ATTN_FWD": "1", "MMFB_ATTN_BWD": "16"}),
    (9, 6, 256, 256, 64, 0.1, {"MMFB_ATTN_BWD": "16"}),
]


@pytest.mark.parametrize("B,heads,Sq,Skv,d,p_drop,env", ATTN_RANDOM)
def test_attention_random_per_element(B, heads, Sq, Skv, d, p_drop, env, monkeypatch):
    """Random inputs: per-element bounds and per-(sample, head) rel-L2 <= 1e-2 for ctx, lse2, dq, dk, dv; dk / dv rows of
    masked keys exactly 0 in every sample with a live key; outputs written into NaN-filled views of larger buffers (an
    element the kernel skips stays NaN), gaps untouched."""
    F, _ = _F()
    for kname, val in env.items():
        monkeypatch.setenv(kname, val)
    g = torch.Generator(device="cuda").manual_seed(B * Sq + Skv + d)
    W = heads * d
    q, k, v, add, mask01, keep, dm, scale = _attn_random(F, B, heads, Sq, Skv, d, g, p_drop)
    out, ob = canary_view((B * Sq, W), torch.bfloat16, 4, 64, fill=NAN)
    ctx, lse2 = F.attention_fwd(q, k, v, B, heads, Sq, Skv, mask=add, drop_mask=dm, drop_scale=scale, out=out)
    dctx = _rand(B * Sq, W, g, 1.0)
    bufs = [canary_view((rows, W), torch.bfloat16, 4, 64, fill=NAN) for rows in (B * Sq, B * Skv, B * Skv)]
    dq, dk, dv = F.attention_bwd(dctx, q, k, v, ctx, lse2, B, heads, Sq, Skv, mask=add, drop_mask=dm, drop_scale=scale,
                                 dq=bufs[0][0], dk=bufs[1][0], dv=bufs[2][0])
    torch.cuda.synchronize()
    for (view, base), name in zip([(out, ob)] + bufs, ("ctx", "dq", "dk", "dv")):
        assert_gaps_untouched(base, view, fill=NAN, name=name)
    rc, bc, rl, bl = attention_fwd_ref_bound(q, k, v, B, heads, Sq, Skv, mask=add, keep=keep, drop_scale=scale)
    r = {"ctx": check_bounded("ctx", ctx, rc, bc), "lse2": check_bounded("lse2", lse2, rl, bl)}
    rdq, rdk, rdv, bdq, bdk, bdv = attention_bwd_ref_bound(q, k, v, dctx, B, heads, Sq, Skv, mask=add, keep=keep,
                                                           drop_scale=scale, ctx_lo=False)
    r.update(dq=check_bounded("dq", dq, rdq, bdq), dk=check_bounded("dk", dk, rdk, bdk), dv=check_bounded("dv", dv, rdv, bdv))
    blk = lambda t, S: t.view(B, S, heads, d)
    for name, got, ref, S in (("ctx", ctx, rc, Sq), ("dq", dq, rdq, Sq), ("dk", dk, rdk, Skv), ("dv", dv, rdv, Skv)):
        # the fully masked sample 0 has a tiny dq / dk (uniform softmax, dS ~ 0): its relative error is not meaningful
        first = 0 if name in ("ctx", "dv") else 1
        r[name + "_head"] = check_blocks(blk(got, S)[first:], blk(ref, S)[first:], (1, S, 1, d), 1e-2, name=name)
    has_live = mask01.sum(1) > 0
    dead = ((mask01 == 0) & has_live[:, None]).reshape(-1)
    for name, t in (("dk", dk), ("dv", dv)):
        # +0 bit for bit (int16 view): a -0 or any stray value in a masked key's gradient row fails
        bits = t[dead].view(torch.int16)
        assert torch.equal(bits, torch.zeros_like(bits)), "%s rows of masked keys must be exactly +0" % name
    _report("attn B%d h%d Sq%d Skv%d d%d p%.1f %s" % (B, heads, Sq, Skv, d, p_drop, env or ""), **r)


@pytest.mark.parametrize("Sq,Skv,d", [(228, 228, 64), (300, 300, 64), (100, 100, 128)])
def test_attention_samples_are_isolated(Sq, Skv, d):
    """Changing sample b+1's keys and values must leave every output of sample b bit-identical."""
    F, _ = _F()
    g = torch.Generator(device="cuda").manual_seed(Sq + d)
    B, heads = 4, 4
    q, k, v, add, mask01, keep, dm, scale = _attn_random(F, B, heads, Sq, Skv, d, g, 0.1, fused=False)
    dctx = _rand(B * Sq, heads * d, g, 1.0)

    def run(k_, v_):
        c, l = F.attention_fwd(q, k_, v_, B, heads, Sq, Skv, mask=add, drop_mask=dm, drop_scale=scale)
        grads = F.attention_bwd(dctx, q, k_, v_, c, l, B, heads, Sq, Skv, mask=add, drop_mask=dm, drop_scale=scale)
        return [c.clone(), l.clone()] + [t.clone() for t in grads]
    first = run(k, v)
    k2, v2 = k.clone(), v.clone()
    k2[2 * Skv:3 * Skv] = _rand(Skv, heads * d, g, 3.0)
    v2[2 * Skv:3 * Skv] = _rand(Skv, heads * d, g, 3.0)
    second = run(k2, v2)
    torch.cuda.synchronize()
    rows_q = slice(0, 2 * Sq)
    rows_k = slice(0, 2 * Skv)
    for name, a, b, rows in zip(("ctx", "lse2", "dq", "dk", "dv"), first, second, (rows_q, None, rows_q, rows_k, rows_k)):
        if rows is None:
            assert torch.equal(a[:2], b[:2]), name
        else:
            assert torch.equal(a[rows], b[rows]), name
    assert not torch.equal(first[0][2 * Sq:3 * Sq], second[0][2 * Sq:3 * Sq])


def test_attention_rejects_misshaped_buffers():
    F, _ = _F()
    B, heads, S, d = 2, 2, 40, 64
    W = heads * d
    q = torch.zeros(B * S, W, dtype=torch.bfloat16, device="cuda")
    big = torch.zeros(B * S + 8, W + 64, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(ValueError):
        F.attention_fwd(q, q, q, B, heads, S, S, out=big[:B * S - 1, :W])
    with pytest.raises(ValueError):
        F.attention_fwd(q, q, q, B, heads, S, S, out=big[:B * S, :W - 8])
    ctx, lse2 = F.attention_fwd(q, q, q, B, heads, S, S)
    for kw in ({"dq": big[:B * S - 1, :W]}, {"dk": big[:B * S, :W - 8]}, {"dv": big[:B * S - 2, :W]}):
        with pytest.raises(ValueError):
            F.attention_bwd(q, q, q, q, ctx, lse2, B, heads, S, S, **kw)
    lbig = torch.zeros(B * heads * S + 64, dtype=torch.float32, device="cuda")
    with pytest.raises(ValueError):
        F.attention_bwd(q, q, q, q, ctx, lbig[:B * heads * (S - 1)].view(B, heads, S - 1), B, heads, S, S)
    torch.cuda.synchronize()


# ======================================================================================================================
# LayerNorm
# ======================================================================================================================
LN_SHAPES = [(M, H) for H in (8, 24, 72, 264, 520, 1032, 1544, 2048) for M in (1, 7, 9, 2369)] + [(37848, 768)]


def _ln_case(F, M, H, with_extra, ld_pad, g):
    y = _rand(M, H, g, 1.0)
    if M > 3:
        y[3] = 0.75                                       # constant row: var = 0, rstd = 1/sqrt(eps)
    y_st, _ = _nan_input(y, pad_cols=ld_pad)
    gamma = (1 + 0.1 * torch.randn(H, generator=g, device="cuda")).to(torch.bfloat16)
    beta = (0.1 * torch.randn(H, generator=g, device="cuda")).to(torch.bfloat16)
    keep = bits = None
    scale = 1.0
    if with_extra:
        keep = torch.rand(M, H, generator=g, device="cuda") >= 0.1
        bits, scale = F.pack_keep_bits(keep), 1 / 0.9
    return y, y_st, gamma, beta, keep, bits, scale


def _ln_run(F, M, H, with_extra, ld_pad, g, fwd=True):
    y, y_st, gamma, beta, keep, bits, scale = _ln_case(F, M, H, with_extra, ld_pad, g)
    r = {}
    out, ob = canary_view((M, H), torch.bfloat16, 2, 8)
    x, mean, rstd = F.layernorm_fwd(y_st, gamma, beta, out=out)
    torch.cuda.synchronize()
    assert_gaps_untouched(ob, out, name="x")
    if fwd:
        rx, rm, rr, bx, bm, br = layernorm_fwd_ref_bound(y, gamma, beta)
        r["x"] = check_bounded("x", x, rx, bx)
        r["mean"] = check_bounded("mean", mean, rm, bm)
        r["rstd"] = check_bounded("rstd", rstd, rr, br)
        if M > 3:
            assert torch.equal(x[3], beta), "a constant row must give exactly beta"
        if keep is not None:                          # the forward's own dropout
            xd, _, _ = F.layernorm_fwd(y_st, gamma, beta, drop_mask=bits, drop_scale=scale)
            rxd, _, _, bxd, _, _ = layernorm_fwd_ref_bound(y, gamma, beta, keep=keep, drop_scale=scale)
            r["x_drop"] = check_bounded("x drop", xd, rxd, bxd)
    dx = _rand(M, H, g, 1.0)
    dx_st, _ = _nan_input(dx, pad_cols=ld_pad)
    dx2 = dx2_st = None
    if with_extra:
        dx2 = _rand(M, H, g, 1.0)
        dx2_st, _ = _nan_input(dx2, pad_cols=ld_pad)
    dgamma = torch.zeros(H, device="cuda")
    dbeta = torch.zeros(H, device="cuda")
    dbias = torch.zeros(H, device="cuda")
    for call in (1, 2):
        dy, dz = F.layernorm_bwd(dx_st, y_st, mean, rstd, gamma, dgamma, dbeta, dbias=dbias, dx2=dx2_st, drop_mask=bits,
                                 drop_scale=scale)
    torch.cuda.synchronize()
    rdy, rdz, bdy, bdz, rdg, bdg, rdb, bdb, rdbias, bdbias = layernorm_bwd_ref_bound(dx, y, gamma, dx2=dx2, keep=keep,
                                                                                    drop_scale=scale)
    r["dy"] = check_bounded("dy", dy, rdy, bdy)
    r["dz"] = check_bounded("dz", dz, rdz, bdz)
    # "a second call accumulates": the buffers hold two calls' worth
    r["dgamma"] = check_bounded("dgamma", dgamma, 2 * rdg, 2 * bdg + 2 * U32 * rdg.abs())
    r["dbeta"] = check_bounded("dbeta", dbeta, 2 * rdb, 2 * bdb + 2 * U32 * rdb.abs())
    r["dbias"] = check_bounded("dbias", dbias, 2 * rdbias, 2 * bdbias + 2 * U32 * rdbias.abs())
    return r


@pytest.mark.parametrize("M,H", LN_SHAPES)
def test_layernorm_per_element(M, H):
    """Every H class (one to eight 256-column vectors, the generic nv = 8 kernels above 1024) at row counts that leave a
    partial warp group and that wrap the grid-stride loop; out= in a sentinel buffer; mean / rstd / dgamma / dbeta / dbias
    against fp64.  Each shape runs twice: plain with row strides H + 64, and with dx2 and dropout (the forward's own keep
    mask as well as the backward's) with row strides H + 8; NaN in every gap."""
    F, _ = _F()
    for with_extra in (False, True):
        g = torch.Generator(device="cuda").manual_seed(M * 4099 + H + with_extra)
        r = _ln_run(F, M, H, with_extra, 8 if with_extra else 64, g)
        assert ("x_drop" in r) == with_extra
        _report("layernorm %dx%d extra=%d" % (M, H, with_extra), **r)


@pytest.mark.parametrize("variant", ["stream", "lean", "tile", "pair"])
@pytest.mark.parametrize("M,H", [(9, 24), (2369, 264), (2369, 520), (7, 1024)])
@pytest.mark.parametrize("with_extra", [False, True])
def test_layernorm_bwd_variants(variant, M, H, with_extra, monkeypatch):
    """The backward variants MMFB_LN_BWD selects per call (H <= 1024), each against fp64 directly."""
    F, _ = _F()
    monkeypatch.setenv("MMFB_LN_BWD", variant)
    g = torch.Generator(device="cuda").manual_seed(M + H + with_extra)
    r = _ln_run(F, M, H, with_extra, 8, g, fwd=False)
    _report("layernorm bwd %s %dx%d extra=%d" % (variant, M, H, with_extra), **r)


def test_layernorm_rejects_misshaped_buffers():
    F, _ = _F()
    M, H = 16, 256
    y = torch.randn(M, H, device="cuda").to(torch.bfloat16)
    vec = torch.ones(2 * H, dtype=torch.bfloat16, device="cuda")
    big = torch.zeros(M + 4, H + 64, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(ValueError):
        F.layernorm_fwd(y, vec[:H - 8], vec[:H])
    with pytest.raises(ValueError):
        F.layernorm_fwd(y, vec[:H], vec[:H - 8])
    with pytest.raises(ValueError):
        F.layernorm_fwd(y, vec[:H], vec[:H], out=big[:M - 1, :H])
    words = torch.zeros(M + 4, 16, dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError):
        F.layernorm_fwd(y, vec[:H], vec[:H], drop_mask=words[:M, :H // 32 - 1])
    x, mean, rstd = F.layernorm_fwd(y, vec[:H], vec[:H])
    f = torch.zeros(2 * H + 64, device="cuda")
    ok = dict(dx=y, y=y, mean=mean, rstd=rstd, gamma=vec[:H], dgamma=f[:H], dbeta=f[H:2 * H])
    for bad in ({"mean": f[:M - 1]}, {"rstd": f[:M - 1]}, {"gamma": vec[:H - 8]}, {"dgamma": f[:H - 8]},
                {"dbeta": f[:H - 8]}, {"dbias": f[:H - 8]}, {"drop_mask": words[:M, :H // 32 - 1]}):
        kw = dict(ok)
        kw.update(bad)
        with pytest.raises(ValueError):
            F.layernorm_bwd(**kw)
    torch.cuda.synchronize()


# ======================================================================================================================
# cross entropy
# ======================================================================================================================
@pytest.mark.parametrize("V", [8, 264, 30528])
def test_ce_rows_per_element(V):
    """row_loss per row against fp64 logsumexp - z_label, d(logits) per element; labels at 0, V - 1 and inside the last
    8-wide vector, ignored rows; a row with one logit at +80 and the rest at -80 gives loss 0 and gradient 0 exactly;
    logits are a column slice of a sentinel buffer."""
    F, _ = _F()
    g = torch.Generator(device="cuda").manual_seed(V)
    M = 37
    z = (torch.randn(M, V, generator=g, device="cuda") * 3).to(torch.bfloat16)
    labels = torch.randint(0, V, (M,), generator=g, device="cuda")
    labels[0], labels[1], labels[2], labels[3], labels[4] = 0, V - 1, V - 3, -1, V - 8
    labels[5] = 2 % V
    z[5] = -80.0
    z[5, 2 % V] = 80.0
    view, base = canary_view((M, V), torch.bfloat16, 2, 8)
    view.copy_(z)
    loss, bl, d, bd = ce_ref_bound(z, labels, 0.125)
    loss_sum = torch.zeros((), device="cuda")
    row_loss = torch.empty(M, device="cuda")
    F.ce_rows(view, labels, -1, 0.125, loss_sum, row_loss=row_loss)
    torch.cuda.synchronize()
    assert_gaps_untouched(base, view, name="logits")
    r = {"row_loss": check_bounded("row_loss", row_loss, loss, bl), "dlogits": check_bounded("dlogits", view, d, bd)}
    r["loss_sum"] = check_bounded("loss_sum", loss_sum, loss.sum(), bl.sum() + M * U32 * loss.abs().sum())
    assert row_loss[5].item() == 0.0 and torch.equal(view[5], torch.zeros_like(view[5]))
    _report("ce_rows V=%d" % V, **r)


def _lce_reference(h, w, b, labels, ignore_index=-1):
    """fp64 loss / dh / dW / db of mean CE(h W^T + b) with bounds that carry the bf16 logits (gemm bound), the ce_rows
    bound on d(logits) and the dgrad / wgrad GEMMs (fp32 accumulation, bf16 dh)."""
    z, bz, _ = gemm_ref_bound(h, w, b)
    active = labels != ignore_index
    n = max(int(active.sum()), 1)
    loss_r, bl, d, bd = ce_ref_bound(z, labels, 1.0 / n, ignore_index)
    p = torch.softmax(z, 1)
    # a logit error dz moves p_j by <= p_j (|dz_j| + sum_k p_k |dz_k|) and the row loss by <= sum_k p_k |dz_k| + |dz_label|
    spz = (p * bz).sum(1, keepdim=True)
    act = active[:, None].double()
    bd = bd + (p * (bz + spz)) / n * act
    lab = labels.clamp_min(0)[:, None]
    bl = bl + (spz.squeeze(1) + bz.gather(1, lab).squeeze(1)) * active.double()
    h64, w64 = h.double(), w.double()
    dh = d @ w64
    bdh = U16 * dh.abs() + bd @ w64.abs() + (w.shape[0] + 2) * U32 * (d.abs() @ w64.abs())
    dw = d.t() @ h64
    bdw = bd.t() @ h64.abs() + (h.shape[0] + 2) * U32 * (d.abs().t() @ h64.abs())
    db = d.sum(0)
    bdb = bd.sum(0) + (h.shape[0] + 2) * U32 * d.abs().sum(0)
    return loss_r.sum() / n, bl.sum() / n + U32 * loss_r.sum() / n, dh, bdh, dw, bdw, db, bdb


def test_linear_cross_entropy_per_element():
    """ops.linear_cross_entropy at V = 30522 (padded to 30528 inside) against fp64: loss, dh, dW, db per element; labels
    include 30521 and ignored rows; chunking over rows with a partial last chunk."""
    from mmf_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(5)
    M, K, V = 300, 128, 30522
    h = _rand(M, K, g, 1.0)
    w = _rand(V, K, g, 0.1)
    b = _rand(1, V, g, 0.1)[0]
    labels = torch.randint(0, V, (M,), generator=g, device="cuda")
    labels[0], labels[1], labels[2] = V - 1, 0, -1
    labels[10:20] = -1
    hp = h.float().requires_grad_(True)
    wp = w.float().requires_grad_(True)
    bp = b.float().requires_grad_(True)
    loss = ops.linear_cross_entropy(hp, wp, bp, labels, ignore_index=-1, chunk_rows=128)
    loss.backward()
    torch.cuda.synchronize()
    rl, bl, dh, bdh, dw, bdw, db, bdb = _lce_reference(h, w, b, labels)
    # the backward hands the fp32 parameter gradients back after one more fp32 scaling by the incoming 1.0
    r = {"loss": check_bounded("loss", loss, rl, bl), "dh": check_bounded("dh", hp.grad, dh, bdh),
         "dW": check_bounded("dW", wp.grad, dw, bdw + U32 * dw.abs()), "db": check_bounded("db", bp.grad, db, bdb + U32 * db.abs())}
    _report("linear_cross_entropy V=%d" % V, **r)
    # every label ignored: loss 0 and zero gradients
    for t in (hp, wp, bp):
        t.grad = None
    loss = ops.linear_cross_entropy(hp, wp, bp, torch.full((M,), -1, device="cuda"), ignore_index=-1)
    loss.backward()
    assert loss.item() == 0.0
    assert all(torch.equal(t.grad, torch.zeros_like(t.grad)) for t in (hp, wp, bp))


@pytest.mark.parametrize("bad", [30522, 30527, -5])
def test_linear_cross_entropy_rejects_labels_outside_the_vocabulary(bad):
    """A label in the vocabulary padding [30522, 30528) or a negative label other than ignore_index is an error, as in
    the reference's CrossEntropyLoss (the fp64 CPU reference raises for the same labels)."""
    from mmf_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(6)
    M, K, V = 16, 64, 30522
    h, w = _rand(M, K, g, 1.0), _rand(V, K, g, 0.1)
    labels = torch.randint(0, V, (M,), generator=g, device="cuda")
    labels[3] = -1
    labels[7] = bad
    with pytest.raises((IndexError, RuntimeError)):
        torch.nn.functional.cross_entropy(h.double().cpu() @ w.double().cpu().t(), labels.cpu(), ignore_index=-1)
    with pytest.raises(ValueError):
        ops.linear_cross_entropy(h, w, None, labels, ignore_index=-1)
    torch.cuda.synchronize()
