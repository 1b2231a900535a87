"""Per-element and per-block comparison helpers for the kernel tests, plus out-of-bounds canaries.

A global relative L2 error averages over the whole output, so one wrong row, one mis-scaled head or one dropped key
can hide under a 1e-2 bar.  These helpers compare every element against an fp64 reference with a bound derived from the
arithmetic the kernel actually does (bf16 operands and outputs, fp32 accumulation), and every block (tile, head, sample)
with its own relative L2 error.  They need no GPU: the references are plain torch in float64 on whatever device the
inputs live on.

Unit roundoffs used in the derivations: fp32 u32 = 2^-24, bf16 u16 = 2^-8 (round to nearest, 8 significant bits).
Summing n fp32 terms in any order is off by at most n * u32 * sum|terms| (first order, Higham 3.1).
"""
import math

import torch

U32 = 2.0 ** -24
U16 = 2.0 ** -8
LN2 = math.log(2.0)
LOG2E = 1.0 / LN2
# fp32 GELU / GELU' of the kernels (mmf_b200/csrc/common.cuh gelu_phi_parts): Abramowitz-Stegun 7.1.26 for erf (|err| <=
# 1.5e-7, so Phi is within 7.5e-8), one ex2.approx and one rcp.approx (<= 2 ulp each) and about 8 fp32 roundings of
# values <= 1.13: at most 7.5e-8 + 12 * 2^-24 = 7.9e-7 < 2^-20 absolute on Phi and on GELU', and |x| times that on GELU
GELU_IMPL = 2.0 ** -20
GELU_GRAD_MAX = 1.13    # max |GELU'(x)| = 1.1289 (at x = +-sqrt(2))


# ----------------------------------------------------------------------------------------------------------------------
# comparisons
# ----------------------------------------------------------------------------------------------------------------------
def check_bounded(name, got, ref64, bound):
    """Assert |got - ref64| <= bound element by element (all float64 after conversion) and that got is finite.
    Returns max(err / bound) so a test can print how much of the bound it used.  On failure the message names the worst
    element: its index, value, reference and bound."""
    g = got.detach().double()
    r = ref64.detach().double()
    b = torch.as_tensor(bound, dtype=torch.float64, device=r.device).expand_as(r)
    if g.shape != r.shape:
        raise AssertionError("%s: shape %s, reference %s" % (name, tuple(g.shape), tuple(r.shape)))
    bad = ~torch.isfinite(g)
    if bad.any():
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError("%s: non-finite value %r at %s (reference %r)" % (name, g[idx].item(), idx, r[idx].item()))
    err = (g - r).abs()
    ratio = err / b.clamp_min(1e-300)
    ratio = torch.where(err == 0, torch.zeros_like(ratio), ratio)
    flat = int(ratio.argmax())
    worst = ratio.reshape(-1)[flat].item()
    if worst > 1.0:
        idx = tuple(int(i) for i in torch.unravel_index(torch.tensor(flat), r.shape))
        n_bad = int((ratio > 1.0).sum())
        raise AssertionError("%s: %d element(s) over the bound; worst at %s: got %.9g, reference %.9g, |err| %.3g > bound %.3g "
                             "(%.2fx)" % (name, n_bad, idx, g[idx].item(), r[idx].item(), err[idx].item(), b[idx].item(),
                                          worst))
    return worst


def block_rel_l2(got, ref, block_shape):
    """Relative L2 error of every block of `block_shape` (a trailing partial block is its own, smaller block).
    Returns a tensor with one entry per block."""
    g = got.detach().double()
    r = ref.detach().double()
    if len(block_shape) != r.dim():
        raise ValueError("block_shape needs one extent per dimension")
    pads = []
    nb = []
    for n, bs in zip(reversed(r.shape), reversed(block_shape)):
        pads += [0, (-n) % bs]
    for n, bs in zip(r.shape, block_shape):
        nb.append((n + bs - 1) // bs)
    d = torch.nn.functional.pad(g - r, pads)
    rr = torch.nn.functional.pad(r, pads)
    shape = []
    for n, bs in zip(nb, block_shape):
        shape += [n, bs]
    d = d.reshape(shape)
    rr = rr.reshape(shape)
    dims = tuple(range(1, 2 * len(nb), 2))
    num = (d * d).sum(dims).sqrt()
    den = (rr * rr).sum(dims).sqrt()
    return num / den.clamp_min(1e-300)


def check_blocks(got, ref, block_shape, tol, name="blocks"):
    """Assert that every block's relative L2 error is <= tol (e.g. per (sample, head) or per 128-row tile instead of
    over the whole tensor).  Returns the worst block's error."""
    e = block_rel_l2(got, ref, block_shape)
    worst = e.max().item()
    if not worst <= tol:
        idx = tuple(int(i) for i in torch.unravel_index(e.argmax(), e.shape))
        raise AssertionError("%s: block %s of shape %s has rel-L2 %.3e > %.1e (%d of %d blocks over)"
                             % (name, idx, tuple(block_shape), worst, tol, int((e > tol).sum()), e.numel()))
    return worst


def global_rel_l2(got, ref):
    g, r = got.detach().double(), ref.detach().double()
    return ((g - r).norm() / r.norm().clamp_min(1e-300)).item()


# ----------------------------------------------------------------------------------------------------------------------
# canaries
# ----------------------------------------------------------------------------------------------------------------------
CANARY_BITS = {torch.bfloat16: 0x7FA5, torch.float32: 0x7FC0DEAD, torch.int32: 0x5A5A5A5A}
_INT_VIEW = {torch.bfloat16: torch.int16, torch.float16: torch.int16, torch.float32: torch.int32, torch.int32: torch.int32,
             torch.float64: torch.int64, torch.int64: torch.int64}


def canary_view(shape, dtype, pad_rows=0, pad_cols=0, fill=None, device="cuda"):
    """A [rows, cols] view inside a [rows + pad_rows, cols + pad_cols] buffer: the view starts pad_rows // 2 rows in, so
    there are gap rows before and after it and pad_cols gap columns after every row (the leading dimension is
    cols + pad_cols).  `fill` is a float (use NaN for inputs: an out-of-bounds read then turns an output non-finite) or
    None for the fixed bit pattern CANARY_BITS[dtype] (use it for outputs: assert_gaps_untouched then finds any write
    outside the view).  Returns (view, base); the view's own elements hold the fill too until written."""
    rows, cols = shape
    lead = pad_rows // 2
    base = torch.empty(rows + pad_rows, cols + pad_cols, dtype=dtype, device=device)
    if fill is None:
        base.view(_INT_VIEW[dtype]).fill_(_as_signed(CANARY_BITS[dtype], _INT_VIEW[dtype]))
    else:
        base.fill_(fill)
    return base[lead:lead + rows, :cols], base


def _as_signed(bits, itype):
    nbits = torch.iinfo(itype).bits
    return bits - (1 << nbits) if bits >= 1 << (nbits - 1) else bits


def gap_mask(base, view):
    """bool mask over base: True where the element lies outside view"""
    if view.untyped_storage().data_ptr() != base.untyped_storage().data_ptr():
        raise ValueError("view does not live in base")
    off = view.storage_offset() - base.storage_offset()
    m = torch.ones(base.numel(), dtype=torch.bool, device=base.device)
    m.as_strided(view.shape, view.stride(), off).fill_(False)
    return m.view(base.shape)


def assert_gaps_untouched(base, view, fill=None, name="output"):
    """Every element of base outside view must still hold its fill, compared bit for bit (fill None = the default
    CANARY_BITS pattern of canary_view).  A write one element past a row or one row past the end fails here."""
    itype = _INT_VIEW[base.dtype]
    bits = base.view(itype)
    if fill is None:
        expect = torch.tensor(_as_signed(CANARY_BITS[base.dtype], itype), dtype=itype, device=base.device)
    else:
        expect = torch.tensor([fill], dtype=base.dtype, device=base.device).view(itype)[0]
    m = gap_mask(base, view)
    changed = m & (bits != expect)
    if changed.any():
        idx = tuple(int(i) for i in changed.nonzero()[0])
        raise AssertionError("%s: %d element(s) outside the view were written, first at base index %s (view starts at row "
                             "%d)" % (name, int(changed.sum()), idx, (view.storage_offset() - base.storage_offset())
                                      // base.stride(0)))


# ----------------------------------------------------------------------------------------------------------------------
# bounds
# ----------------------------------------------------------------------------------------------------------------------
def gemm_ref_bound(a, b, bias=None, out_bf16=True):
    """fp64 reference r = A B^T (+ bias) and its per-element bound, for bf16 A [M, K], B [N, K] and fp32 accumulation.

    The kernel sums K exact bf16 x bf16 products in fp32 (error <= K u32 (|A||B|^T)_ij), adds the bias in fp32 (one more
    rounding of a value <= |A||B|^T + |bias|), and rounds once to bf16 (<= u16 |value|).  So
        |got - r| <= u16 |r| + (1 + u16) (K + 2) u32 ((|A||B|^T)_ij + |bias_j|)
    Without out_bf16 (the fp32 wgrad epilogue) the u16 |r| term becomes u32 |r| (red.global adds into a zeroed fp32
    buffer: one more rounding).  Returns (r, bound, acc_bound) where acc_bound is the fp32 part alone."""
    a64, b64 = a.double(), b.double()
    r = a64 @ b64.t()
    mag = a64.abs() @ b64.abs().t()
    if bias is not None:
        r = r + bias.double()
        mag = mag + bias.double().abs()
    K = a.shape[1]
    acc = (K + 2) * U32 * mag
    rnd = U16 if out_bf16 else U32
    return r, rnd * r.abs() + (1 + rnd) * acc, acc


def gelu64(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def gelu_grad64(x):
    return 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


def epi_bound_gelu(u_ref, u_acc_bound):
    """GELU of the fp32 pre-activation u: |Δh| <= u16 |h| + (1 + u16) (max|GELU'| |Δu| + GELU_IMPL |u|), where |Δu| is u's
    fp32 error (the bf16 u output is rounded separately; h is computed from the fp32 value)."""
    h = gelu64(u_ref)
    return h, U16 * h.abs() + (1 + U16) * (GELU_GRAD_MAX * u_acc_bound + GELU_IMPL * (u_ref.abs() + u_acc_bound))


def epi_bound_gelu_bwd(acc_ref, acc_bound, x):
    """du = acc * GELU'(x) with x bf16 exact: |Δdu| <= u16 |du| + (1 + u16) (|GELU'(x)| Δacc + |acc| (GELU_IMPL + u32))"""
    gp = gelu_grad64(x.double())
    r = acc_ref * gp
    return r, U16 * r.abs() + (1 + U16) * (gp.abs() * acc_bound + (acc_ref.abs() + acc_bound) * (GELU_IMPL + U32))


def attention_fwd_ref_bound(q, k, v, B, heads, Sq, Skv, mask=None, keep=None, drop_scale=1.0):
    """fp64 ctx [B*Sq, W] and lse2 [B, heads, Sq] (log2 of the softmax denominator, in the kernels' base-2 units) with
    per-element bounds, for bf16 q [B*Sq, W], k/v [B*Skv, W], additive fp32 mask [B, Skv], bool keep [B, h, Sq, Skv].

    The kernels compute s2 = (q.k) * log2(e)/sqrt(d) + mask * log2(e) in fp32 (d products: error <= d u32 (|q||k|) per
    score, plus about two roundings of |s2| and of the row max m), p = ex2.approx(s2 - m) (<= 2 ulp), round p to bf16 for
    the P.V MMA (u16 relative per key), sum the p of the row in fp32 for the denominator l and divide at the end.  With
    e_ij = ln2 (d u32 |q||k|_ij log2(e)/sqrt(d) + 2 u32 (|s2_ij| + |m_i|)) + 2^-22 the relative error of one unnormalised p
    and P_ij the fp64 probabilities (times keep * scale with dropout), the first-order error of ctx_i is
        numerator:   sum_j P_ij |v_j| (u16 + e_ij + Skv u32)     (bf16 P, score error, fp32 accumulation of Skv terms)
        denominator: |ctx_i| (u16 + max_j e_ij + Skv u32)        (l carries the same per-key errors; u16 covers a kernel
                                                                  that sums the bf16-rounded p)
        output:      u16 |ctx_i|                                 (bf16 store)
    and lse2 = m + log2(l) is within (max_j e_ij + Skv u32) / ln2 + 4 u32 |lse2|."""
    W = q.shape[-1]
    d = W // heads
    q4 = q.double().view(B, Sq, heads, d).transpose(1, 2)
    k4 = k.double().view(B, Skv, heads, d).transpose(1, 2)
    v4 = v.double().view(B, Skv, heads, d).transpose(1, 2)
    c2 = LOG2E / math.sqrt(d)
    s2 = (q4 @ k4.transpose(-1, -2)) * c2
    if mask is not None:
        s2 = s2 + mask.double().view(B, 1, 1, Skv) * LOG2E
    m = s2.amax(-1, keepdim=True)
    p = torch.exp2(s2 - m)
    l = p.sum(-1, keepdim=True)
    P = p / l
    Pd = P * keep.double() * drop_scale if keep is not None else P
    ctx = Pd @ v4
    mag = (q4.abs() @ k4.abs().transpose(-1, -2)) * c2
    e = LN2 * (d * U32 * mag + 2 * U32 * (s2.abs() + m.abs())) + 2.0 ** -22
    num = (Pd * (U16 + e + Skv * U32)) @ v4.abs()
    emax = e.amax(-1, keepdim=True)
    bound = num + ctx.abs() * (2 * U16 + emax + Skv * U32)
    lse2 = (m + torch.log2(l)).squeeze(-1)
    lse_bound = (emax.squeeze(-1) + Skv * U32) / LN2 + 4 * U32 * lse2.abs()
    merge = lambda t: t.transpose(1, 2).reshape(B * t.shape[2], W)
    return merge(ctx), merge(bound), lse2, lse_bound


def attention_bwd_ref_bound(q, k, v, dctx, B, heads, Sq, Skv, mask=None, keep=None, drop_scale=1.0, ctx_lo=True):
    """fp64 dq, dk, dv ([B*S, W]) and per-element bounds for the recompute backward.

    With P, Pd as in attention_fwd_ref_bound, dO = dctx, dP = dO V^T (times keep * scale), delta_i = rowsum(dO_i * O_i) and
    dS = P (dP - delta):  dv_j = sum_i Pd_ij dO_i,  dk_j = (1/sqrt(d)) sum_i dS_ij q_i,  dq_i = (1/sqrt(d)) sum_j dS_ij k_j.
    The backward recomputes p_ij = exp2(s2_ij - lse2_i) with the forward's lse2, so one P_ij is within
        e_ij = e0_ij + max_k e0_ik + Skv u32 + 4 ln2 u32 |lse2_i|
    relative: its own score / ex2 error e0_ij (as in attention_fwd_ref_bound) plus ln2 times the lse2 bound derived there.
    delta_i is summed in fp32 over the forward's stored ctx (d + 2 roundings), whose per-element error is the forward bound
        ΔO = sum_j Pd_ij |v_j| (u16 + e0_ij + Skv u32) + |O_i| (u16 + max_j e0_ij + Skv u32) + r |O_i|
    with r = u16 for the bf16 ctx alone (ctx_lo=False) and r = u16^2 when the bf16 residual ctx_lo restores the fp32 value,
    so Δdelta_i = sum_d |dO_i| ΔO_i + (d + 2) u32 sum_d |dO_i O_i|.  The kernels feed bf16-rounded Pd and dS to the MMAs
    and accumulate in fp32.  Error of one dS_ij:
        |ΔdS_ij| <= P_ij (|dP_ij - delta_i| (u16 + e_ij) + d u32 (|dO||V|^T)_ij + Δdelta_i)
    and then, with u16 |x| for every bf16 output x,
        |Δdv_j| <= u16 |dv_j| + sum_i Pd_ij (u16 + e_ij + Sq u32) |dO_i|
        |Δdk_j| <= u16 |dk_j| + (1/sqrt(d)) sum_i (|ΔdS_ij| + (u16 + Sq u32) |dS_ij|) |q_i|
        |Δdq_i| <= u16 |dq_i| + (1/sqrt(d)) sum_j (|ΔdS_ij| + (u16 + Skv u32) |dS_ij|) |k_j|"""
    W = q.shape[-1]
    d = W // heads
    sh = lambda t, S: t.double().view(B, S, heads, d).transpose(1, 2)
    q4, k4, v4, do4 = sh(q, Sq), sh(k, Skv), sh(v, Skv), sh(dctx, Sq)
    c = 1.0 / math.sqrt(d)
    s2 = (q4 @ k4.transpose(-1, -2)) * (c * LOG2E)
    if mask is not None:
        s2 = s2 + mask.double().view(B, 1, 1, Skv) * LOG2E
    m = s2.amax(-1, keepdim=True)
    p = torch.exp2(s2 - m)
    P = p / p.sum(-1, keepdim=True)
    kd = keep.double() * drop_scale if keep is not None else None
    Pd = P * kd if kd is not None else P
    O = Pd @ v4
    dP = do4 @ v4.transpose(-1, -2)
    dPmag = do4.abs() @ v4.abs().transpose(-1, -2)
    if kd is not None:
        dP, dPmag = dP * kd, dPmag * kd
    mag = (q4.abs() @ k4.abs().transpose(-1, -2)) * (c * LOG2E)
    e0 = LN2 * (d * U32 * mag + 2 * U32 * (s2.abs() + m.abs())) + 2.0 ** -22
    e0max = e0.amax(-1, keepdim=True)
    lse2 = m + torch.log2(p.sum(-1, keepdim=True))
    e = e0 + e0max + Skv * U32 + 4 * LN2 * U32 * lse2.abs()
    O_err = ((Pd * (U16 + e0 + Skv * U32)) @ v4.abs() + O.abs() * (U16 + e0max + Skv * U32)
              + O.abs() * (U16 * U16 if ctx_lo else U16))
    delta = (do4 * O).sum(-1, keepdim=True)
    ddelta = (do4.abs() * O_err).sum(-1, keepdim=True) + (d + 2) * U32 * (do4 * O).abs().sum(-1, keepdim=True)
    dS = P * (dP - delta)
    edS = P * ((dP - delta).abs() * (U16 + e) + d * U32 * dPmag + ddelta)
    dv = Pd.transpose(-1, -2) @ do4
    dk = c * (dS.transpose(-1, -2) @ q4)
    dq = c * (dS @ k4)
    bdv = U16 * dv.abs() + (Pd * (U16 + e + Sq * U32)).transpose(-1, -2) @ do4.abs()
    bdk = U16 * dk.abs() + c * ((edS + (U16 + Sq * U32) * dS.abs()).transpose(-1, -2) @ q4.abs())
    bdq = U16 * dq.abs() + c * ((edS + (U16 + Skv * U32) * dS.abs()) @ k4.abs())
    merge = lambda t: t.transpose(1, 2).reshape(B * t.shape[2], W)
    return tuple(merge(t) for t in (dq, dk, dv, bdq, bdk, bdv))


def layernorm_fwd_ref_bound(y, gamma, beta, eps=1e-12, keep=None, drop_scale=1.0):
    """fp64 x = (LN(y) * gamma + beta) [* keep * scale], mean, rstd and bounds, for bf16 y [M, H].

    fp32 in the kernel: mean of H bf16 values (error <= H u32 mean|y|), variance of the centred values (the stable
    two-pass form; relative error <= (H + 4) u32), rsqrt (<= 2 ulp): rstd relative error e_r = (H + 8) u32 / 2 + 2 u32 and
    |Δmean| = H u32 mean|y|.  Then x = (y - mean) rstd gamma + beta in fp32 and one bf16 rounding:
        |Δx| <= u16 |x| + (1 + u16) (|gamma| rstd (|Δmean| + |y - mean| e_r) + 4 u32 (|x̂ gamma| + |beta|))
    (times keep * scale with dropout).  Returns (x, mean, rstd, bound_x, bound_mean, bound_rstd)."""
    y64 = y.double()
    H = y.shape[1]
    mean = y64.mean(1)
    var = ((y64 - mean[:, None]) ** 2).mean(1)
    rstd = 1.0 / torch.sqrt(var + eps)
    xh = (y64 - mean[:, None]) * rstd[:, None]
    g, b = gamma.double(), beta.double()
    x = xh * g + b
    # H copies of one bf16 value (8 significant bits) sum exactly in fp32 for H <= 2^16: a constant row has an exact mean
    dmean = torch.where(var > 0, H * U32 * y64.abs().mean(1), torch.zeros_like(var))
    # a zero-variance row has rstd = 1/sqrt(eps) and centred values that are exactly 0 in the kernel as well
    er = torch.where(var > 0, torch.full_like(var, (H + 8) * U32 / 2 + 2 * U32) + dmean * 2 *
                     (y64 - mean[:, None]).abs().mean(1) / var.clamp_min(1e-300), torch.full_like(var, 4 * U32))
    bx = U16 * x.abs() + (1 + U16) * (g.abs() * rstd[:, None] * (dmean[:, None] + (y64 - mean[:, None]).abs() * er[:, None])
                                      + 4 * U32 * ((xh * g).abs() + b.abs()))
    if keep is not None:
        kd = keep.double() * drop_scale
        x, bx = x * kd, bx * kd + U32 * (x * kd).abs()
    return x, mean, rstd, bx, dmean, rstd * er


def layernorm_bwd_ref_bound(dx, y, gamma, eps=1e-12, dx2=None, keep=None, drop_scale=1.0):
    """fp64 dy, dz (per element) and dgamma, dbeta, dbias (per column) with bounds, for the LayerNorm backward that
    reads the kernel's own fp32 mean / rstd (whose errors layernorm_fwd_ref_bound bounds: |Δmean|, rstd e_r).

    g = (dx + dx2) gamma (fp32, exact up to one rounding), x̂ = (y - mean) rstd, a = mean(g), c = mean(g x̂):
        dy = rstd (g - a - x̂ c),  dz = dy * keep * scale,  dgamma = sum_rows (dx + dx2) x̂,  dbeta = sum_rows (dx + dx2),
        dbias = sum_rows dz.
    fp32 means over H terms are within H u32 of the mean of magnitudes; x̂ is within |x̂| e_r + rstd |Δmean|:
        |Δdy| <= u16 |dy| + (1 + u16) (rstd ((H + 4) u32 (|g| + mean|g| + |x̂| mean|g x̂|) + Δx̂ (|c| + mean|g|))
                                       + |dy| e_r)
        |Δdgamma_j| <= M u32 sum|(dx + dx2) x̂| + sum |dx + dx2| Δx̂,   |Δdbeta_j| <= (M + 1) u32 sum |dx + dx2|
        |Δdbias_j| <= sum_rows bound(dz) + M u32 sum |dz|  (the row/column kernel pair sums the stored bf16 dz)."""
    M, H = y.shape
    y64 = y.double()
    mean = y64.mean(1, keepdim=True)
    var = ((y64 - mean) ** 2).mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    xh = (y64 - mean) * rstd
    dsum = dx.double() + (dx2.double() if dx2 is not None else 0.0)
    g = dsum * gamma.double()
    a = g.mean(1, keepdim=True)
    c = (g * xh).mean(1, keepdim=True)
    dy = rstd * (g - a - xh * c)
    dmean = torch.where(var > 0, H * U32 * y64.abs().mean(1, keepdim=True), torch.zeros_like(var))
    er = torch.where(var > 0, (H + 8) * U32 / 2 + 2 * U32 + dmean * 2 * (y64 - mean).abs().mean(1, keepdim=True)
                     / var.clamp_min(1e-300), torch.full_like(var, 4 * U32))
    dxh = xh.abs() * er + rstd * dmean
    bdy = U16 * dy.abs() + (1 + U16) * (rstd * ((H + 4) * U32 * (g.abs() + g.abs().mean(1, keepdim=True)
                                                                + xh.abs() * (g * xh).abs().mean(1, keepdim=True))
                                                + dxh * (c.abs() + g.abs().mean(1, keepdim=True)))
                                        + dy.abs() * er)
    if keep is not None:
        kd = keep.double() * drop_scale
        dz, bdz = dy * kd, bdy * kd + U16 * (dy * kd).abs()
    else:
        dz, bdz = dy, bdy
    dgamma = (dsum * xh).sum(0)
    bdg = M * U32 * (dsum * xh).abs().sum(0) + (dsum.abs() * dxh).sum(0)
    dbeta = dsum.sum(0)
    bdb = (M + 1) * U32 * dsum.abs().sum(0)
    dbias = dz.sum(0)
    bdbias = bdz.sum(0) + (M + 1) * U32 * dz.abs().sum(0)
    return dy, dz, bdy, bdz, dgamma, bdg, dbeta, bdb, dbias, bdbias


def ce_ref_bound(z, labels, grad_scale, ignore_index=-1):
    """fp64 row loss (logsumexp(z) - z[label], 0 for ignored rows) and d(logits) = (softmax - onehot) grad_scale with
    bounds, for bf16 logits z [M, V].

    The kernel takes the row max mx, sums p_j = ex2.approx(z_j log2(e) - mx log2(e)) in fp32 and divides.  One p_j is
    within e_j = 2^-21 + 2 ln2 u32 (|z_j| + |mx|) log2(e) relative (the ex2 error and the roundings of its argument), the
    sum within e = max_j e_j + V u32.  So
        |Δloss| <= e + 3 u32 (|mx| + |log sum| + |z_label|)
        |Δd_j| <= u16 |d_j| + (1 + u16) grad_scale (p_j (e_j + e + 2 u32) + u32 [j = label] + 2^-126)."""
    z64 = z.double()
    M, V = z.shape
    lab = labels.to(torch.int64)
    active = (lab != ignore_index) & (lab >= 0) & (lab < V)
    safe = torch.where(active, lab, torch.zeros_like(lab))
    mx = z64.amax(1, keepdim=True)
    ez = torch.exp(z64 - mx)
    s = ez.sum(1, keepdim=True)
    p = ez / s
    lse = (mx + torch.log(s)).squeeze(1)
    zl = z64.gather(1, safe[:, None]).squeeze(1)
    loss = torch.where(active, lse - zl, torch.zeros_like(lse))
    ej = 2.0 ** -21 + 2 * LN2 * U32 * (z64.abs() + mx.abs()) * LOG2E
    e = ej.amax(1, keepdim=True) + V * U32
    onehot = torch.zeros_like(z64).scatter_(1, safe[:, None], 1.0)
    d = (p - onehot) * grad_scale
    # plus 2^-126: a p below the smallest normal fp32 number may flush to zero (ex2.approx.ftz)
    bd = U16 * d.abs() + (1 + U16) * grad_scale * (p * (ej + e + 2 * U32) + U32 * onehot + 2.0 ** -126)
    act = active[:, None].double()
    bloss = (e.squeeze(1) + 3 * U32 * (mx.squeeze(1).abs() + torch.log(s).squeeze(1).abs() + zl.abs())) * active.double()
    return loss, bloss, d * act, bd * act
