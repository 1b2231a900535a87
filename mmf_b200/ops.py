"""Differentiable building blocks over the C-ABI kernels, for the front-ends around the encoder trunk
(MMBT modal embeddings, MMFTransformer per-modality embeddings, ViLBERT image embeddings).

Unlike the encoder/VisualBERT-embedding fast path (flat parameter pack, one autograd node per module), these are
ordinary `torch.autograd.Function`s taking the parameters as inputs: the front-ends are a few percent of the block's
FLOPs, so flexibility wins over launch count.  All arithmetic still runs in libmmfb200 kernels; activations bf16.
"""
import torch

from . import functional as F
from . import lib
from .engine import best_splits


def _bf16(t):
    return t.detach().to(torch.bfloat16).contiguous()


class _Linear(torch.autograd.Function):
    """y = x W^T + b on the tcgen05 GEMM; backward: dgrad (MN-major W), split-K wgrad, column-sum bias gradient."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        xb, wb = _bf16(x), _bf16(weight)
        bb = _bf16(bias) if bias is not None else None
        y = F.gemm(xb, wb, epi=lib.EPI_BIAS, bias=bb)
        ctx.save_for_backward(xb, wb)
        ctx.dtypes = (x.dtype, weight.dtype, bias.dtype if bias is not None else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        xb, wb = ctx.saved_tensors
        dyb = dy.to(torch.bfloat16).contiguous()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = F.gemm(dyb, wb, b_mn=True, epi=lib.EPI_BIAS).to(ctx.dtypes[0])
        if ctx.needs_input_grad[1]:
            dw = torch.zeros(wb.shape, dtype=torch.float32, device=wb.device)
            F.gemm(dyb, xb, a_mn=True, b_mn=True, epi=lib.EPI_ATOMIC_F32, out=dw,
                   splits=best_splits(wb.shape[0], wb.shape[1], xb.shape[0]))
            dw = dw.to(ctx.dtypes[1])
        if ctx.dtypes[2] is not None and ctx.needs_input_grad[2]:
            db = torch.zeros(wb.shape[0], dtype=torch.float32, device=wb.device)
            F.colsum(dyb, db)
            db = db.to(ctx.dtypes[2])
        return dx, dw, db


def linear(x2d, weight, bias=None):
    """x2d [M, K] (any float dtype) -> bf16 [M, N].  K and N must be multiples of 8 (TMA row pitch)."""
    return _Linear.apply(x2d, weight, bias)


class _LinearReLU(torch.autograd.Function):
    """y = relu(x W^T + b): GEMM with the ReLU epilogue; backward masks dy with (y > 0) and reuses the Linear backward."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        xb, wb, bb = _bf16(x), _bf16(weight), _bf16(bias)
        y = F.gemm(xb, wb, epi=lib.EPI_BIAS_RELU, bias=bb)
        ctx.save_for_backward(xb, wb, y)
        ctx.dtypes = (x.dtype, weight.dtype, bias.dtype)
        return y

    @staticmethod
    def backward(ctx, dy):
        xb, wb, y = ctx.saved_tensors
        dz = F.relu_bwd(dy.to(torch.bfloat16).contiguous(), y)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = F.gemm(dz, wb, b_mn=True, epi=lib.EPI_BIAS).to(ctx.dtypes[0])
        if ctx.needs_input_grad[1]:
            dw = torch.zeros(wb.shape, dtype=torch.float32, device=wb.device)
            F.gemm(dz, xb, a_mn=True, b_mn=True, epi=lib.EPI_ATOMIC_F32, out=dw,
                   splits=best_splits(wb.shape[0], wb.shape[1], xb.shape[0]))
            dw = dw.to(ctx.dtypes[1])
        if ctx.needs_input_grad[2]:
            db = torch.zeros(wb.shape[0], dtype=torch.float32, device=wb.device)
            F.colsum(dz, db)
            db = db.to(ctx.dtypes[2])
        return dx, dw, db


def linear_relu(x2d, weight, bias):
    return _LinearReLU.apply(x2d, weight, bias)


class _LinearGELU(torch.autograd.Function):
    """h = gelu(x W^T + b): GEMM with the bias + GELU epilogue (it also writes the pre-activation u, saved for the
    backward); backward: du = dh * GELU'(u) (row kernel), then the Linear backward."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        xb, wb, bb = _bf16(x), _bf16(weight), _bf16(bias)
        u, h = F.gemm(xb, wb, epi=lib.EPI_BIAS_GELU, bias=bb)
        ctx.save_for_backward(xb, wb, u)
        ctx.dtypes = (x.dtype, weight.dtype, bias.dtype)
        return h

    @staticmethod
    def backward(ctx, dh):
        xb, wb, u = ctx.saved_tensors
        du = F.gelu_bwd(dh.to(torch.bfloat16).contiguous(), u)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = F.gemm(du, wb, b_mn=True, epi=lib.EPI_BIAS).to(ctx.dtypes[0])
        if ctx.needs_input_grad[1]:
            dw = torch.zeros(wb.shape, dtype=torch.float32, device=wb.device)
            F.gemm(du, xb, a_mn=True, b_mn=True, epi=lib.EPI_ATOMIC_F32, out=dw,
                   splits=best_splits(wb.shape[0], wb.shape[1], xb.shape[0]))
            dw = dw.to(ctx.dtypes[1])
        if ctx.needs_input_grad[2]:
            db = torch.zeros(wb.shape[0], dtype=torch.float32, device=wb.device)
            F.colsum(du, db)
            db = db.to(ctx.dtypes[2])
        return dx, dw, db


def linear_gelu(x2d, weight, bias):
    return _LinearGELU.apply(x2d, weight, bias)


class _LayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps):
        xb, g, b = _bf16(x), _bf16(weight), _bf16(bias)
        y, mean, rstd = F.layernorm_fwd(xb, g, b, eps)
        ctx.save_for_backward(xb, mean, rstd, g)
        ctx.dtypes = (x.dtype, weight.dtype, bias.dtype)
        return y

    @staticmethod
    def backward(ctx, dy):
        xb, mean, rstd, g = ctx.saved_tensors
        dg = torch.zeros(g.shape, dtype=torch.float32, device=g.device)
        db = torch.zeros_like(dg)
        dx, _ = F.layernorm_bwd(dy.to(torch.bfloat16).contiguous(), xb, mean, rstd, g, dg, db)
        return dx.to(ctx.dtypes[0]), dg.to(ctx.dtypes[1]), db.to(ctx.dtypes[2]), None


def layer_norm(x2d, weight, bias, eps=1e-12):
    return _LayerNorm.apply(x2d, weight, bias, eps)


class _ComposeLN(torch.autograd.Function):
    """out = dropout(LN(sum_k src_k[rows_k] + sum_k table_k[idx_k]))  - the embedding composer + LayerNorm.

    inputs: n_src dense sources then n_tab tables then (ln_w, ln_b); index tensors are int32 [M] (negative = absent).
    """

    @staticmethod
    def forward(ctx, meta, *tensors):
        M, H, n_src, n_tab, rows, idxs, eps, bits, scale = meta
        srcs = [_bf16(t) for t in tensors[:n_src]]
        tabs = [_bf16(t) for t in tensors[n_src:n_src + n_tab]]
        g, b = _bf16(tensors[-2]), _bf16(tensors[-1])
        y = F.embed_compose(M, H, srcs=list(zip(srcs, rows)), tabs=list(zip(tabs, idxs[0])), device=g.device)
        x, mean, rstd = F.layernorm_fwd(y, g, b, eps, drop_mask=bits, drop_scale=scale)
        ctx.meta = meta
        ctx.src_shapes = [tuple(t.shape) for t in srcs]
        ctx.tab_shapes = [tuple(t.shape) for t in tabs]
        ctx.dtypes = [t.dtype for t in tensors]
        ctx.save_for_backward(y, mean, rstd, g)
        return x

    @staticmethod
    def backward(ctx, dout):
        M, H, n_src, n_tab, rows, idxs, eps, bits, scale = ctx.meta
        y, mean, rstd, g = ctx.saved_tensors
        d = dout.to(torch.bfloat16).contiguous()
        if bits is not None:   # dropout sits after the LayerNorm
            d = (d * F.unpack_keep_bits(bits, H) * scale).to(torch.bfloat16)
        dg = torch.zeros(H, dtype=torch.float32, device=g.device)
        db = torch.zeros_like(dg)
        dy, _ = F.layernorm_bwd(d, y, mean, rstd, g, dg, db)
        dsrcs = [torch.zeros(s, dtype=torch.bfloat16, device=g.device) for s in ctx.src_shapes]
        dtabs = [torch.zeros(s, dtype=torch.float32, device=g.device) for s in ctx.tab_shapes]
        if dsrcs:
            F.embed_scatter(dy, dsrcs=list(zip(dsrcs, rows)))
        for t, ix in zip(dtabs, idxs[1]):
            F.embed_scatter_sorted(dy, t, *F.sort_indices(ix))   # idxs already carry -1 at padding_idx rows
        grads = [t.to(dt) for t, dt in zip(dsrcs + dtabs + [dg, db], ctx.dtypes)]
        return (None,) + tuple(grads)


def compose_ln(M, H, srcs, tabs, ln_weight, ln_bias, eps=1e-12, p=0.0, training=False, dropout_state=None):
    """srcs: up to 2 (tensor [*, H], int32 rows [M]); tabs: up to 3 (table [V, H], int32 idx [M][, padding_idx]).
    The same table may appear in several slots.  Returns bf16 [M, H]."""
    if len(srcs) > 2 or len(tabs) > 3:
        raise ValueError("compose_ln: at most 2 dense sources and 3 table slots")
    bits, scale = None, 1.0
    if training and p > 0.0:
        from .modules import _fresh_dropout_state
        ds = dropout_state or _fresh_dropout_state()
        bits, scale = ds.bits((M,), H, p, ln_weight.device), 1.0 / (1.0 - p)
    # a table slot may be (table, idx, padding_idx): the row is read in the forward but, like nn.Embedding(padding_idx=),
    # receives no gradient - the backward index gets -1 (= absent) there
    fwd_idx = [t[1] for t in tabs]
    bwd_idx = [t[1] if len(t) < 3 or t[2] is None else torch.where(t[1] == t[2], torch.full_like(t[1], -1), t[1])
               for t in tabs]
    meta = (M, H, len(srcs), len(tabs), [r for _, r in srcs], (fwd_idx, bwd_idx), float(eps), bits, scale)
    return _ComposeLN.apply(meta, *[t for t, _ in srcs], *[t[0] for t in tabs], ln_weight, ln_bias)


def i32(t):
    return t.reshape(-1).to(torch.int32).contiguous()


def linear_any(x2d, weight, bias=None):
    """`linear` for arbitrary out/in feature counts: the GEMM wants N and K in multiples of 8 (16-byte TMA row pitch), so a
    classifier with 2 labels or a 5-column location input gets zero-padded operands and a sliced result; autograd's
    pad / slice backward routes the gradients.  No-op wrapper when the sizes already fit."""
    N, K = weight.shape
    pn, pk = (-N) % 8, (-K) % 8
    if pk:
        x2d = torch.nn.functional.pad(x2d, (0, pk))
        weight = torch.nn.functional.pad(weight, (0, pk))
    if pn:
        weight = torch.nn.functional.pad(weight, (0, 0, 0, pn))
        if bias is not None:
            bias = torch.nn.functional.pad(bias, (0, pn))
    y = linear(x2d, weight, bias)
    return y[:, :N] if pn else y


class _LinearCrossEntropy(torch.autograd.Function):
    """mean cross-entropy of (h W^T + b) against integer labels WITHOUT the [rows, V] logits tensor: the rows are processed
    in chunks - vocabulary GEMM -> mmfb_ce_rows (loss + d(logits) in place) -> dgrad and split-K wgrad of the chunk - so at
    most `chunk_rows` x V logits exist at a time (sized to stay L2-resident between the three kernels that touch them).
    Gradients are therefore computed in the FORWARD (scaled by 1 / n_active); the backward multiplies them by the incoming
    scalar.  Reference: prediction scores + CrossEntropyLoss(ignore_index) of mmf/models/visual_bert.py:269-277 and
    mmf/models/transformers/heads/mlm.py:83-88."""

    @staticmethod
    def forward(ctx, h, weight, bias, labels, ignore_index, chunk_rows):
        hb, wb = _bf16(h), _bf16(weight)
        V, K = wb.shape
        pad = (-V) % 8
        if pad:                                # V = 30522 is not a multiple of 8: zero rows, and a -inf-like bias so that
            wb = torch.nn.functional.pad(wb, (0, 0, 0, pad))      # the padded logits vanish from the softmax
        bb = _bf16(bias) if bias is not None else torch.zeros(V, dtype=torch.bfloat16, device=wb.device)
        if pad:
            bb = torch.cat([bb, torch.full((pad,), -30000.0, dtype=torch.bfloat16, device=bb.device)])
        M = hb.shape[0]
        labels = labels.reshape(-1).to(torch.int64).contiguous()
        # the one host read of the head (the reference's mean reduction) also carries the count of labels outside [0, V):
        # the kernel would score a label in the vocabulary padding against a pad column and silently drop a negative one,
        # where the reference's CrossEntropyLoss raises
        active = labels != ignore_index
        n_active, n_bad = torch.stack([active.sum(), (active & ((labels < 0) | (labels >= V))).sum()]).tolist()
        if n_bad:
            raise ValueError("linear_cross_entropy: %d label(s) outside [0, %d) that are not ignore_index (%d)"
                             % (n_bad, V, ignore_index))
        scale = 1.0 / float(max(n_active, 1))
        loss_sum = torch.zeros((), dtype=torch.float32, device=wb.device)
        need_h, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        need_b = bias is not None and ctx.needs_input_grad[2]
        dh = torch.empty_like(hb) if need_h else None
        dw = torch.zeros(wb.shape, dtype=torch.float32, device=wb.device) if need_w else None
        db = torch.zeros(wb.shape[0], dtype=torch.float32, device=wb.device) if need_b else None
        for r0 in range(0, M, chunk_rows):
            r1 = min(M, r0 + chunk_rows)
            z = F.gemm(hb[r0:r1], wb, epi=lib.EPI_BIAS, bias=bb)
            F.ce_rows(z, labels[r0:r1], ignore_index, scale, loss_sum)      # z now holds d(logits)
            if need_h:
                F.gemm(z, wb, b_mn=True, epi=lib.EPI_BIAS, out=dh[r0:r1])
            if need_w:
                F.gemm(z, hb[r0:r1], a_mn=True, b_mn=True, epi=lib.EPI_ATOMIC_F32, out=dw,
                       splits=best_splits(wb.shape[0], K, r1 - r0))
            if need_b:
                F.colsum(z, db)
        ctx.save_for_backward(*[t for t in (dh, dw, db) if t is not None])
        ctx.have = (need_h, need_w, need_b)
        ctx.V = V
        ctx.dtypes = (h.dtype, weight.dtype, bias.dtype if bias is not None else None)
        return loss_sum * scale

    @staticmethod
    def backward(ctx, g):
        saved = list(ctx.saved_tensors)
        need_h, need_w, need_b = ctx.have
        dh = saved.pop(0) if need_h else None
        dw = saved.pop(0) if need_w else None
        db = saved.pop(0) if need_b else None
        gh = (dh.float() * g).to(ctx.dtypes[0]) if need_h else None
        gw = (dw[:ctx.V] * g).to(ctx.dtypes[1]) if need_w else None
        gb = (db[:ctx.V] * g).to(ctx.dtypes[2]) if need_b else None
        return gh, gw, gb, None, None, None


def linear_cross_entropy(h2d, weight, bias, labels, ignore_index=-1, chunk_rows=2048):
    """mean_i CE((h W^T + b)_i, labels_i) over the rows with labels_i != ignore_index (0 when there is none), fp32 scalar."""
    return _LinearCrossEntropy.apply(h2d, weight, bias, labels, int(ignore_index), int(chunk_rows))
