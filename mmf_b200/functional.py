"""Thin Python wrappers over the C ABI: one function per exported kernel entry point.

Each wrapper validates dtypes/devices, allocates outputs with torch (so the caching allocator and
autograd own every buffer) and enqueues the kernel on the current CUDA stream.  Nothing here
computes on the CPU.
"""
import ctypes

import torch

from . import lib
from .lib import LIB, AdamWArgs, AttnArgs, ComposeArgs, GemmArgs, LnArgs, ScatterArgs, _ptr, _stream_ptr, check


def _req(t, dtype, name):
    if t is None:
        return
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: the B200 path has no CPU fallback" % name)
    if t.dtype != dtype:
        raise ValueError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if t.stride(-1) != 1:
        raise ValueError("%s must be contiguous in its last dimension" % name)


def _idx_len(idx, M, name):
    """the kernels read one index per output row and never check: a short index buffer is an out-of-bounds device read"""
    if idx.numel() != M or not idx.is_contiguous():
        raise ValueError("%s must be a contiguous vector of %d indices (one per row), got shape %s" % (name, M, tuple(idx.shape)))


def _shape(t, shape, name, contiguous=False):
    """the kernels take a pointer and a row stride and trust the extents: a buffer smaller than the problem is an
    out-of-bounds device access (a vector, or a buffer read with an implied stride, must also be contiguous)"""
    if t is None:
        return
    if tuple(t.shape) != tuple(shape) or (contiguous and not t.is_contiguous()):
        raise ValueError("%s must be %s%s, got shape %s%s" % (name, "a contiguous " if contiguous else "", list(shape),
                                                               list(t.shape), "" if t.is_contiguous() else " (strided)"))


def gemm(a, b, *, a_mn=False, b_mn=False, epi=lib.EPI_BIAS, bias=None, aux=None, drop_mask=None,
         drop_scale=1.0, out=None, out2=None, splits=1, block_n=0, cluster=0):
    """C[M,N] = epi(A[M,K] @ B[N,K]^T) on the tcgen05 GEMM.

    a: [M,K] (a_mn=False) or [K,M] (a_mn=True); b: [N,K] (b_mn=False) or [K,N] (b_mn=True); bf16.
    Returns C (and C2 for EPI_BIAS_GELU).  For EPI_ATOMIC_F32 `out` (fp32 [M,N]) is accumulated into.
    """
    _req(a, torch.bfloat16, "a")
    _req(b, torch.bfloat16, "b")
    _req(bias, torch.bfloat16, "bias")
    _req(aux, torch.bfloat16, "aux")
    if a.dim() != 2 or b.dim() != 2:
        raise ValueError("gemm operands must be 2-D")
    M, K = (a.shape[1], a.shape[0]) if a_mn else (a.shape[0], a.shape[1])
    N, Kb = (b.shape[1], b.shape[0]) if b_mn else (b.shape[0], b.shape[1])
    if K != Kb:
        raise ValueError("gemm: inner dimensions differ (%d vs %d)" % (K, Kb))
    if epi == lib.EPI_ATOMIC_F32:
        if out is None:
            out = torch.zeros(M, N, dtype=torch.float32, device=a.device)
        _req(out, torch.float32, "out")
    else:
        if out is None:
            out = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
        _req(out, torch.bfloat16, "out")
        if epi == lib.EPI_BIAS_GELU and out2 is None:
            # the kernel stores C2 with C's row stride: give the default C2 the same one
            out2 = torch.empty(M, max(out.stride(0), N), dtype=torch.bfloat16, device=a.device)[:, :N]
    _shape(out, (M, N), "gemm: out")
    if out2 is not None:
        _req(out2, torch.bfloat16, "out2")
        _shape(out2, (M, N), "gemm: out2")
        if out2.stride(0) != out.stride(0):
            raise ValueError("gemm: out2 must have the row stride of out (%d), got %d" % (out.stride(0), out2.stride(0)))
    _shape(bias, (N,), "gemm: bias", contiguous=True)
    _shape(aux, (M, N), "gemm: aux")
    args = GemmArgs()
    args.A, args.lda, args.a_mn = a.data_ptr(), a.stride(0), int(a_mn)
    args.B, args.ldb, args.b_mn = b.data_ptr(), b.stride(0), int(b_mn)
    args.C, args.ldc = out.data_ptr(), out.stride(0)
    args.C2 = out2.data_ptr() if out2 is not None else None
    args.bias = bias.data_ptr() if bias is not None else None
    args.aux, args.ldaux = (aux.data_ptr(), aux.stride(0)) if aux is not None else (None, 0)
    if drop_mask is not None:
        _req(drop_mask, torch.int32, "drop_mask")
        _shape(drop_mask, (M, (N + 31) // 32), "gemm: drop_mask")
        args.drop_mask, args.ldmask = drop_mask.data_ptr(), drop_mask.stride(0)
    args.drop_scale = float(drop_scale)
    args.M, args.N, args.K = M, N, K
    args.epi, args.splits, args.block_n, args.cluster = int(epi), int(splits), int(block_n), int(cluster)
    check(LIB.mmfb_gemm(ctypes.byref(args), _stream_ptr()))
    if epi == lib.EPI_BIAS_GELU:
        return out, out2
    return out


def _attn_args(q, k, v, B, heads, Sq, Skv, mask, drop_mask, drop_scale):
    for t, n in ((q, "q"), (k, "k"), (v, "v")):
        _req(t, torch.bfloat16, n)
    W = q.shape[-1]
    if W % heads:
        raise ValueError(
            "The hidden size (%d) is not a multiple of the number of attention heads (%d)" % (W, heads))
    if q.shape[0] != B * Sq or k.shape[0] != B * Skv or v.shape[0] != B * Skv:
        raise ValueError("attention: q/k/v row counts do not match B*Sq / B*Skv")
    a = AttnArgs()
    a.q, a.ldq = q.data_ptr(), q.stride(0)
    a.k, a.ldk = k.data_ptr(), k.stride(0)
    a.v, a.ldv = v.data_ptr(), v.stride(0)
    if mask is not None:
        _req(mask, torch.float32, "mask")
        if tuple(mask.shape) != (B, Skv) or not mask.is_contiguous():
            raise ValueError("attention: additive mask must be contiguous fp32 [B, Skv]")
        a.mask = mask.data_ptr()
    if drop_mask is not None:
        _req(drop_mask, torch.int32, "drop_mask")
        if tuple(drop_mask.shape) != (B, heads, Sq, (Skv + 31) // 32) or not drop_mask.is_contiguous():
            raise ValueError("attention: drop_mask must be contiguous int32 [B, heads, Sq, ceil(Skv/32)]")
        a.drop_mask, a.drop_scale = drop_mask.data_ptr(), float(drop_scale)
    a.B, a.heads, a.Sq, a.Skv, a.head_dim = B, heads, Sq, Skv, W // heads
    return a


def attention_fwd(q, k, v, B, heads, Sq, Skv, mask=None, drop_mask=None, drop_scale=1.0, out=None, save_lo=False):
    """ctx, lse2 (, ctx_lo) = fused softmax(QK^T/sqrt(d) + mask) V.  q [B*Sq, h*d], k/v [B*Skv, h*d] (views allowed).
    save_lo: also return ctx_lo = bf16(O - float(ctx)), the part of the fp32 output the bf16 ctx drops; the backward's
    delta = rowsum(dO * (ctx + ctx_lo)) then carries no common rounding bias per row."""
    a = _attn_args(q, k, v, B, heads, Sq, Skv, mask, drop_mask, drop_scale)
    W = q.shape[-1]
    ctx = out if out is not None else torch.empty(B * Sq, W, dtype=torch.bfloat16, device=q.device)
    _req(ctx, torch.bfloat16, "out")
    _shape(ctx, (B * Sq, W), "attention_fwd: out")
    lse2 = torch.empty(B, heads, Sq, dtype=torch.float32, device=q.device)
    a.ctx, a.ldo, a.lse2 = ctx.data_ptr(), ctx.stride(0), lse2.data_ptr()
    ctx_lo = None
    if save_lo:
        ctx_lo = torch.empty(B * Sq, W, dtype=torch.bfloat16, device=q.device)
        a.ctx_lo = ctx_lo.data_ptr()
    check(LIB.mmfb_attention_fwd(ctypes.byref(a), _stream_ptr()))
    if save_lo:
        return ctx, lse2, ctx_lo
    return ctx, lse2


def attention_bwd(dctx, q, k, v, ctx, lse2, B, heads, Sq, Skv, mask=None, drop_mask=None, drop_scale=1.0,
                  dq=None, dk=None, dv=None, ctx_lo=None):
    """dq, dk, dv from the saved q, k, v, ctx and row statistics (probabilities are recomputed)."""
    a = _attn_args(q, k, v, B, heads, Sq, Skv, mask, drop_mask, drop_scale)
    _req(dctx, torch.bfloat16, "dctx")
    _req(ctx, torch.bfloat16, "ctx")
    W = q.shape[-1]
    _shape(dctx, (B * Sq, W), "attention_bwd: dctx")
    _shape(ctx, (B * Sq, W), "attention_bwd: ctx")
    _req(lse2, torch.float32, "lse2")
    _shape(lse2, (B, heads, Sq), "attention_bwd: lse2", contiguous=True)
    dq = dq if dq is not None else torch.empty(B * Sq, W, dtype=torch.bfloat16, device=q.device)
    dk = dk if dk is not None else torch.empty(B * Skv, W, dtype=torch.bfloat16, device=q.device)
    dv = dv if dv is not None else torch.empty(B * Skv, W, dtype=torch.bfloat16, device=q.device)
    for t, n, rows in ((dq, "dq", B * Sq), (dk, "dk", B * Skv), (dv, "dv", B * Skv)):
        _req(t, torch.bfloat16, n)
        _shape(t, (rows, W), "attention_bwd: " + n)
    delta = torch.empty(B, heads, Sq, dtype=torch.float32, device=q.device)
    a.ctx, a.ldo, a.lse2 = ctx.data_ptr(), ctx.stride(0), lse2.data_ptr()
    a.dctx, a.ld_dctx, a.delta = dctx.data_ptr(), dctx.stride(0), delta.data_ptr()
    if ctx_lo is not None:
        _req(ctx_lo, torch.bfloat16, "ctx_lo")
        if not ctx_lo.is_contiguous() or tuple(ctx_lo.shape) != (B * Sq, W):
            raise ValueError("ctx_lo must be contiguous [B*Sq, heads*head_dim]")
        a.ctx_lo = ctx_lo.data_ptr()
    a.dq, a.ld_dq = dq.data_ptr(), dq.stride(0)
    a.dk, a.ld_dk = dk.data_ptr(), dk.stride(0)
    a.dv, a.ld_dv = dv.data_ptr(), dv.stride(0)
    check(LIB.mmfb_attention_bwd(ctypes.byref(a), _stream_ptr()))
    return dq, dk, dv


def pack_keep_bits(keep):
    """bool [..., n] -> int32 [..., ceil(n/32)] keep-bit words (bit j of word w = element 32*w + j)."""
    n = keep.shape[-1]
    pad = (-n) % 32
    if pad:
        keep = torch.nn.functional.pad(keep, (0, pad))
    k = keep.reshape(*keep.shape[:-1], -1, 32).to(torch.int64)
    weights = (1 << torch.arange(32, device=keep.device, dtype=torch.int64))
    words = (k * weights).sum(-1)
    words = torch.where(words >= 2 ** 31, words - 2 ** 32, words)
    return words.to(torch.int32).contiguous()


LN_EPS = 1e-12


def layernorm_fwd(y, gamma, beta, eps=LN_EPS, drop_mask=None, drop_scale=1.0, out=None):
    """x, mean, rstd = LayerNorm(y) over the last dim; y bf16 [M,H] (row stride allowed)."""
    _req(y, torch.bfloat16, "y"); _req(gamma, torch.bfloat16, "gamma"); _req(beta, torch.bfloat16, "beta")
    M, H = y.shape
    _shape(gamma, (H,), "layernorm_fwd: gamma", contiguous=True)
    _shape(beta, (H,), "layernorm_fwd: beta", contiguous=True)
    x = out if out is not None else torch.empty(M, H, dtype=torch.bfloat16, device=y.device)
    _req(x, torch.bfloat16, "out")
    _shape(x, (M, H), "layernorm_fwd: out")
    mean = torch.empty(M, dtype=torch.float32, device=y.device)
    rstd = torch.empty(M, dtype=torch.float32, device=y.device)
    a = LnArgs()
    a.y, a.ldy, a.gamma, a.beta = y.data_ptr(), y.stride(0), gamma.data_ptr(), beta.data_ptr()
    a.x, a.ldx, a.mean, a.rstd = x.data_ptr(), x.stride(0), mean.data_ptr(), rstd.data_ptr()
    if drop_mask is not None:
        _req(drop_mask, torch.int32, "drop_mask")
        _shape(drop_mask, (M, (H + 31) // 32), "layernorm_fwd: drop_mask")
        a.drop_mask, a.ldmask, a.drop_scale = drop_mask.data_ptr(), drop_mask.stride(0), float(drop_scale)
    a.eps, a.M, a.H = float(eps), M, H
    check(LIB.mmfb_layernorm_fwd(ctypes.byref(a), _stream_ptr()))
    return x, mean, rstd


def layernorm_bwd(dx, y, mean, rstd, gamma, dgamma, dbeta, dbias=None, dx2=None, drop_mask=None, drop_scale=1.0,
                  need_dz=True):
    """Returns (dy, dz): dy = grad wrt y (goes to the residual branch), dz = grad wrt the dense output that was
    dropped before the residual add (dz is dy when there is no dropout).  dgamma/dbeta/dbias (fp32 [H]) are
    accumulated in place."""
    _req(dx, torch.bfloat16, "dx"); _req(y, torch.bfloat16, "y"); _req(gamma, torch.bfloat16, "gamma")
    M, H = y.shape
    _shape(dx, (M, H), "layernorm_bwd: dx")
    _shape(dx2, (M, H), "layernorm_bwd: dx2")
    _shape(gamma, (H,), "layernorm_bwd: gamma", contiguous=True)
    for name, t in (("mean", mean), ("rstd", rstd)):
        _req(t, torch.float32, name)
        _shape(t, (M,), "layernorm_bwd: " + name, contiguous=True)
    dy = torch.empty(M, H, dtype=torch.bfloat16, device=y.device)
    a = LnArgs()
    a.dx, a.lddx = dx.data_ptr(), dx.stride(0)
    if dx2 is not None:
        _req(dx2, torch.bfloat16, "dx2")
        a.dx2, a.lddx2 = dx2.data_ptr(), dx2.stride(0)
    a.y, a.ldy, a.mean, a.rstd, a.gamma = y.data_ptr(), y.stride(0), mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr()
    a.dy, a.lddy = dy.data_ptr(), dy.stride(0)
    dz = dy
    if drop_mask is not None:
        _req(drop_mask, torch.int32, "drop_mask")
        _shape(drop_mask, (M, (H + 31) // 32), "layernorm_bwd: drop_mask")
        dz = torch.empty(M, H, dtype=torch.bfloat16, device=y.device)
        a.drop_mask, a.ldmask, a.drop_scale = drop_mask.data_ptr(), drop_mask.stride(0), float(drop_scale)
    a.dz, a.lddz = dz.data_ptr(), dz.stride(0)
    for name, t in (("dgamma", dgamma), ("dbeta", dbeta), ("dbias", dbias)):
        if t is not None:
            _req(t, torch.float32, name)
            _shape(t, (H,), "layernorm_bwd: " + name, contiguous=True)
            setattr(a, name, t.data_ptr())
    a.M, a.H = M, H
    check(LIB.mmfb_layernorm_bwd(ctypes.byref(a), _stream_ptr()))
    return dy, dz


def colsum(x, out):
    """out[n] += sum_m x[m,n] (x bf16 [M,N], out fp32 [N])."""
    _req(x, torch.bfloat16, "x"); _req(out, torch.float32, "out")
    check(LIB.mmfb_colsum(x.data_ptr(), x.stride(0), out.data_ptr(), x.shape[0], x.shape[1], _stream_ptr()))
    return out


_DROPOUT_EPOCH = {}      # device index -> int64 [1] step counter in device memory (set by mmf_b200.graphs)


def dropout_epoch(device, create=False):
    """The device-resident step counter mixed into every keep-bit draw on `device` once it exists (None otherwise).
    A CUDA-graph capture freezes the host-side (seed, offset) of each draw; the captured graph increments this counter,
    so every replay still draws fresh masks (mmf_b200/graphs.py)."""
    idx = torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    if idx not in _DROPOUT_EPOCH and create:
        _DROPOUT_EPOCH[idx] = torch.zeros(1, dtype=torch.int64, device=torch.device("cuda", idx))
    return _DROPOUT_EPOCH.get(idx)


def dropout_bits(shape_rows, ncols, p, seed, offset, device):
    """int32 keep-bit words [*shape_rows, ceil(ncols/32)] for nn.Dropout(p)."""
    words = (ncols + 31) // 32
    out = torch.empty(*shape_rows, words, dtype=torch.int32, device=device)
    epoch = dropout_epoch(out.device)
    if epoch is None:
        check(LIB.mmfb_dropout_bits(out.data_ptr(), out.numel(), int(seed) & (2 ** 64 - 1), int(offset), float(p),
                                    _stream_ptr()))
    else:
        check(LIB.mmfb_dropout_bits_epoch(out.data_ptr(), out.numel(), int(seed) & (2 ** 64 - 1), int(offset),
                                          epoch.data_ptr(), float(p), _stream_ptr()))
    return out


def relu_bwd(dy, y):
    """dz = dy where y > 0 else 0 (bf16, contiguous)."""
    _req(dy, torch.bfloat16, "dy"); _req(y, torch.bfloat16, "y")
    if not (dy.is_contiguous() and y.is_contiguous()) or dy.numel() != y.numel():
        raise ValueError("relu_bwd: contiguous, equally sized buffers required")
    dz = torch.empty_like(dy)
    check(LIB.mmfb_relu_bwd(dy.data_ptr(), y.data_ptr(), dz.data_ptr(), dy.numel(), _stream_ptr()))
    return dz


def ce_rows(logits, labels, ignore_index, grad_scale, loss_sum, row_loss=None):
    """In place: logits [M, V] bf16 (V % 8 == 0, row stride allowed) -> d(logits) = (softmax - onehot) * grad_scale, zeros for
    rows whose label is ignore_index; the summed loss of the active rows is ADDED to loss_sum (fp32 scalar tensor)."""
    _req(logits, torch.bfloat16, "logits"); _req(labels, torch.int64, "labels")
    if not loss_sum.is_cuda or loss_sum.dtype != torch.float32 or loss_sum.numel() != 1:
        raise ValueError("ce_rows: loss_sum must be a CUDA fp32 tensor with one element")
    M, V = logits.shape
    if labels.numel() != M or not labels.is_contiguous():
        raise ValueError("ce_rows: one contiguous int64 label per row required")
    rl = None
    if row_loss is not None:
        _req(row_loss, torch.float32, "row_loss")
        _shape(row_loss, (M,), "ce_rows: row_loss", contiguous=True)
        rl = row_loss.data_ptr()
    check(LIB.mmfb_ce_rows(logits.data_ptr(), logits.stride(0), labels.data_ptr(), int(ignore_index), M, V, float(grad_scale),
                           loss_sum.data_ptr(), rl, _stream_ptr()))
    return logits


def add(a, b):
    """a + b (bf16, contiguous, same size)."""
    _req(a, torch.bfloat16, "a"); _req(b, torch.bfloat16, "b")
    if not (a.is_contiguous() and b.is_contiguous()) or a.numel() != b.numel():
        raise ValueError("add: contiguous, equally sized buffers required")
    out = torch.empty_like(a)
    check(LIB.mmfb_add_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), a.numel(), _stream_ptr()))
    return out


def dropout_apply(x, drop_mask, drop_scale):
    """keep-bit ? x * scale : 0 for x bf16 [M, H] and keep-bit words int32 [M, ceil(H/32)]."""
    _req(x, torch.bfloat16, "x"); _req(drop_mask, torch.int32, "drop_mask")
    M, H = x.shape
    out = torch.empty(M, H, dtype=torch.bfloat16, device=x.device)
    check(LIB.mmfb_dropout_apply(x.data_ptr(), x.stride(0), drop_mask.data_ptr(), drop_mask.stride(0), float(drop_scale),
                                 out.data_ptr(), out.stride(0), M, H, _stream_ptr()))
    return out


def gelu_bwd(dh, u):
    """du = dh * GELU'(u) (bf16, contiguous) - for a GELU that is followed by a LayerNorm instead of a GEMM."""
    _req(dh, torch.bfloat16, "dh"); _req(u, torch.bfloat16, "u")
    if not (dh.is_contiguous() and u.is_contiguous()) or dh.numel() != u.numel():
        raise ValueError("gelu_bwd: contiguous, equally sized buffers required")
    du = torch.empty_like(dh)
    check(LIB.mmfb_gelu_bwd(dh.data_ptr(), u.data_ptr(), du.data_ptr(), dh.numel(), _stream_ptr()))
    return du


def adamw(param, grad, exp_avg, exp_avg_sq, groups, *, beta1, beta2, eps, mode, grad_scale=1.0, group_of_block=None,
          param_bf16=None):
    """One fused AdamW step over flat fp32 buffers (staged, include/mmfb200.h: mmfb_adamw).
    groups: list (<= 8) of dicts {lr, weight_decay, step_size, bc2_sqrt}; group_of_block: uint8 [n/8] or None."""
    for t, n in ((param, "param"), (grad, "grad"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        _req(t, torch.float32, n)
        if not t.is_contiguous() or t.numel() != param.numel():
            raise ValueError("adamw: %s must be contiguous and as large as param" % n)
    a = AdamWArgs()
    a.param, a.grad, a.exp_avg, a.exp_avg_sq = param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr()
    if param_bf16 is not None:
        _req(param_bf16, torch.bfloat16, "param_bf16")
        a.param_bf16 = param_bf16.data_ptr()
    if group_of_block is not None:
        _req(group_of_block, torch.uint8, "group_of_block")
        if group_of_block.numel() != param.numel() // 8:
            raise ValueError("adamw: group_of_block needs one entry per 8 elements")
        a.group = group_of_block.data_ptr()
    a.n, a.n_groups = param.numel(), len(groups)
    if not 1 <= len(groups) <= 8:
        raise ValueError("adamw: between 1 and 8 hyper-parameter groups per launch")
    for i, g in enumerate(groups):
        a.lr[i], a.weight_decay[i], a.step_size[i], a.bc2_sqrt[i] = g["lr"], g["weight_decay"], g["step_size"], g["bc2_sqrt"]
    a.beta1, a.beta2, a.eps, a.grad_scale, a.mode = float(beta1), float(beta2), float(eps), float(grad_scale), int(mode)
    check(LIB.mmfb_adamw(ctypes.byref(a), _stream_ptr()))


def cast_f32_bf16(src, dst):
    _req(src, torch.float32, "src"); _req(dst, torch.bfloat16, "dst")
    if src.numel() != dst.numel() or not src.is_contiguous() or not dst.is_contiguous():
        raise ValueError("cast: buffers must be contiguous and equally sized")
    check(LIB.mmfb_cast_f32_bf16(src.data_ptr(), dst.data_ptr(), src.numel(), _stream_ptr()))
    return dst


def embed_compose(M, H, srcs=(), tabs=(), device=None):
    """y[r] = sum_k src_k[row_k[r]] + sum_k tab_k[idx_k[r]].
    srcs: up to 2 of (bf16 [*,H] tensor, int32 [M] rows); tabs: up to 3 of (bf16 [V,H] table, int32 [M] idx).
    Negative indices drop the term for that row."""
    a = ComposeArgs()
    keep = []
    for k, (t, rows) in enumerate(srcs):
        _req(t, torch.bfloat16, "src%d" % k); _req(rows, torch.int32, "src_row%d" % k)
        _idx_len(rows, M, "src_row%d" % k)
        a.src[k], a.ldsrc[k], a.src_row[k] = t.data_ptr(), t.stride(0), rows.data_ptr()
        device = t.device
    for k, (t, idx) in enumerate(tabs):
        _req(t, torch.bfloat16, "tab%d" % k); _req(idx, torch.int32, "tab_idx%d" % k)
        _idx_len(idx, M, "tab_idx%d" % k)
        if t.shape[1] != H or not t.is_contiguous():
            raise ValueError("embedding table %d must be contiguous [V, %d]" % (k, H))
        a.tab[k], a.tab_idx[k] = t.data_ptr(), idx.data_ptr()
        device = t.device
    y = torch.empty(M, H, dtype=torch.bfloat16, device=device)
    a.y, a.ldy, a.M, a.H = y.data_ptr(), y.stride(0), M, H
    check(LIB.mmfb_embed_compose(ctypes.byref(a), _stream_ptr()))
    return y


def embed_scatter(dy, dsrcs=(), dtabs=()):
    """Backward of embed_compose: dsrcs (bf16 tensor, rows) get plain row stores, dtabs (fp32 table grad, idx) get
    atomic accumulation."""
    _req(dy, torch.bfloat16, "dy")
    M, H = dy.shape
    a = ScatterArgs()
    for k, (t, rows) in enumerate(dsrcs):
        _req(t, torch.bfloat16, "dsrc%d" % k)
        _idx_len(rows, M, "src_row%d" % k)
        a.dsrc[k], a.ldsrc[k], a.src_row[k] = t.data_ptr(), t.stride(0), rows.data_ptr()
    for k, (t, idx) in enumerate(dtabs):
        _req(t, torch.float32, "dtab%d" % k)
        _idx_len(idx, M, "tab_idx%d" % k)
        a.dtab[k], a.tab_idx[k] = t.data_ptr(), idx.data_ptr()
    a.dy, a.lddy, a.M, a.H = dy.data_ptr(), dy.stride(0), M, H
    check(LIB.mmfb_embed_scatter(ctypes.byref(a), _stream_ptr()))


def sort_indices(idx):
    """(sorted_idx, order) int32 for embed_scatter_sorted; a stable device sort of the [M] index vector."""
    sorted_idx, order = torch.sort(idx.to(torch.int64), stable=True)
    return sorted_idx.to(torch.int32).contiguous(), order.to(torch.int32).contiguous()


def embed_scatter_sorted(dy, dtab, sorted_idx, order):
    """dtab[sorted_idx[k]] += dy[order[k]] with run aggregation (fp32 table gradient)."""
    _req(dy, torch.bfloat16, "dy"); _req(dtab, torch.float32, "dtab")
    _req(sorted_idx, torch.int32, "sorted_idx"); _req(order, torch.int32, "order")
    M, H = dy.shape
    _idx_len(sorted_idx, M, "sorted_idx"); _idx_len(order, M, "order")
    check(LIB.mmfb_embed_scatter_sorted(dy.data_ptr(), dy.stride(0), order.data_ptr(), sorted_idx.data_ptr(),
                                        dtab.data_ptr(), M, H, _stream_ptr()))


def unpack_keep_bits(words, n):
    """int32 [..., W] -> bool [..., n] (test helper / oracle interop; runs on the words' device)."""
    w = words.to(torch.int64) & 0xFFFFFFFF
    bits = (w.unsqueeze(-1) >> torch.arange(32, device=words.device, dtype=torch.int64)) & 1
    return bits.reshape(*words.shape[:-1], -1)[..., :n].bool()
