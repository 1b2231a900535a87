"""End-to-end parity of the B200 encoders (forward + backward through autograd) against
  (1) the reference's own outputs/gradients stored in tests/golden (fp32 reference vs bf16 kernels), and
  (2) the oracle run in fp32 on the same device with the same bf16-rounded weights, at config-2 shapes.
Tolerances: per BASELINE.md 5 the bf16 bar is 1e-2 per layer against the fp32 oracle; end-to-end the reference's own
bf16-vs-fp32 drift is 1.25e-2 (outputs) / 1.8e-2 (gradients) at 12 layers, which is the bound used for deep stacks."""
import types

import pytest
import torch

from oracle import fusion_oracle as O
from oracle import golden_io

pytestmark = pytest.mark.gpu


def rel(a, b, floor=1e-3):
    fl = floor * (b.numel() ** 0.5)
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().norm().clamp_min(fl)).item()


def check_param_grads(named_params, ref_grads, tol, skip=(), drift=None, k=1.5):
    """relative-L2 per parameter; the key bias gradient is analytically zero (softmax is shift invariant), so it
    is only required to be tiny next to the query bias gradient.  `drift` (optional): per-parameter error of the
    reference arithmetic itself when cast to bf16 - BASELINE.md 5: end to end the new path must be no worse than
    the reference's own bf16 drift, so the bound is max(tol, k * drift) with k = 1.5, or 2.5 on the 10-token golden
    fixture where a single draw of rounding noise is not averaged over tokens (at S=228 every parameter passes 2e-2)."""
    worst, worst_n, bad = 0.0, "", []
    named = dict(named_params)
    for n, p in named.items():
        if n in skip:
            continue
        if ".key.bias" in n or ".key1.bias" in n or ".key2.bias" in n:
            qn = n.replace("key", "query")
            assert p.grad.float().norm() <= 0.05 * named[qn].grad.float().norm() + 1e-3, n
            continue
        e = rel(p.grad, ref_grads[n])
        if e > worst:
            worst, worst_n = e, n
        bound = tol if drift is None else max(tol, k * drift.get(n, 0.0))
        if e >= bound:
            bad.append((n, e, bound))
    assert not bad, bad[:8]
    return worst, worst_n


def bert_cfg(hidden, heads, inter, layers, p=0.0):
    return types.SimpleNamespace(hidden_size=hidden, num_attention_heads=heads, intermediate_size=inter,
                                 num_hidden_layers=layers, hidden_dropout_prob=p, attention_probs_dropout_prob=p,
                                 layer_norm_eps=1e-12, hidden_act="gelu", initializer_range=0.02)


def test_bert_encoder_vs_reference_golden():
    from mmf_b200.modules import B200BertEncoder
    g = golden_io.load("bert_encoder")
    c = g["cfg"]
    enc = B200BertEncoder(bert_cfg(c["hidden"], c["heads"], c["inter"], c["layers"]))
    assert set(enc.state_dict().keys()) == set(g["state_dict"].keys())  # checkpoint-key compatibility
    enc.load_state_dict(g["state_dict"])
    enc = enc.cuda().eval()
    x = g["x"].cuda().requires_grad_(True)
    add = O.extended_attention_mask(g["mask"].cuda())
    out = enc(x, add)[0]
    (out * g["w_rand"].cuda()).sum().backward()
    torch.cuda.synchronize()
    e_out, e_dx = rel(out.cpu(), g["out"]), rel(x.grad.cpu(), g["dx"])
    print("golden bert: out %.2e dx %.2e" % (e_out, e_dx))
    assert torch.isfinite(out).all()
    assert e_out < 1e-2 and e_dx < 1e-2            # measured 6.0e-3 / 6.3e-3 (2 layers, 10-token fixture)
    worst, wn = check_param_grads(enc.named_parameters(), g["grads"], 2e-2)
    print("golden bert: worst param-grad rel %.2e (%s)" % (worst, wn))


def test_vilbert_encoder_vs_reference_golden():
    from mmf_b200.modules import B200ViLBertEncoder
    g = golden_io.load("vilbert_encoder")
    c = dict(g["cfg"])
    cfg = types.SimpleNamespace(hidden_dropout_prob=0.0, v_hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                                v_attention_probs_dropout_prob=0.0, **c)
    enc = B200ViLBertEncoder(cfg)
    assert set(enc.state_dict().keys()) == set(g["state_dict"].keys())
    enc.load_state_dict(g["state_dict"])
    enc = enc.cuda().eval()
    txt = g["txt"].cuda().requires_grad_(True)
    img = g["img"].cuda().requires_grad_(True)
    tadd = O.extended_attention_mask(g["tmask"].cuda())
    iadd = O.extended_attention_mask(g["imask"].cuda())
    tl, vl, _ = enc(txt, img, tadd, tadd, iadd, None, output_all_encoded_layers=False)
    ((tl[-1] * g["wt"].cuda()).sum() + (vl[-1] * g["wv"].cuda()).sum()).backward()
    torch.cuda.synchronize()
    errs = {"t_out": rel(tl[-1].cpu(), g["t_out"]), "v_out": rel(vl[-1].cpu(), g["v_out"]),
            "dtxt": rel(txt.grad.cpu(), g["dtxt"]), "dimg": rel(img.grad.cpu(), g["dimg"])}
    print("golden vilbert:", " ".join("%s=%.2e" % kv for kv in errs.items()))
    assert max(errs.values()) < 1.5e-2
    for n, p in enc.named_parameters():
        if n in g["unused"]:
            assert p.grad is None, n   # q_dense1/q_dense2 never receive gradients (vilbert.py:486-494)
    # the reference arithmetic itself in bf16 (oracle with bf16 weights / activations) vs its fp32 golden
    sdb = {k: v.cuda().to(torch.bfloat16).requires_grad_(True) for k, v in g["state_dict"].items()}
    tb = g["txt"].cuda().to(torch.bfloat16).requires_grad_(True)
    ib = g["img"].cuda().to(torch.bfloat16).requires_grad_(True)
    to, vo = O.vilbert_encoder(tb, ib, tadd.to(torch.bfloat16), iadd.to(torch.bfloat16), sdb, "", c)
    ((to.float() * g["wt"].cuda()).sum() + (vo.float() * g["wv"].cuda()).sum()).backward()
    drift = {k: rel(v.grad, g["grads"][k]) for k, v in sdb.items() if v.grad is not None and k in g["grads"]}
    print("golden vilbert: reference-in-bf16 drift: max %.2e" % max(drift.values()))
    worst, wn = check_param_grads(enc.named_parameters(), g["grads"], 2e-2, skip=g["unused"], drift=drift, k=2.5)
    print("golden vilbert: worst param-grad rel %.2e (%s), bf16-reference drift there %.2e" % (worst, wn, drift[wn]))


def _oracle_run(sd, x, add, layers, heads, w_rand, masks=None, p=0.0):
    sdf = {k: v.detach().float().clone().requires_grad_(True) for k, v in sd.items()}
    xf = x.detach().float().clone().requires_grad_(True)
    out = O.bert_encoder(xf, add, sdf, "", layers, heads, masks, p, p)
    (out * w_rand).sum().backward()
    return out.detach(), xf.grad, {k: v.grad for k, v in sdf.items()}


@pytest.mark.parametrize("B,S,H,heads,I,L", [(4, 228, 768, 12, 3072, 2), (2, 122, 768, 12, 3072, 1),
                                             (3, 120, 1024, 16, 4096, 1)])
def test_bert_encoder_vs_oracle_config_shapes(B, S, H, heads, I, L):
    """config 2 (VisualBERT 228 tokens), config 1 (MMBT 122 tokens, 1 layer), config 5 (1024/16h/4096) shapes."""
    from mmf_b200.modules import B200BertEncoder
    torch.manual_seed(0)
    enc = B200BertEncoder(bert_cfg(H, heads, I, L)).cuda().eval()
    with torch.no_grad():   # make biases / LN params non-trivial
        for n, p in enc.named_parameters():
            if p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.02)
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(B, S, H, generator=g, device="cuda")
    lens = torch.randint(S // 2, S + 1, (B,), generator=g, device="cuda")
    mask = (torch.arange(S, device="cuda")[None] < lens[:, None]).long()
    add = O.extended_attention_mask(mask)
    w_rand = torch.randn(B, S, H, generator=g, device="cuda")
    xg = x.clone().requires_grad_(True)
    out = enc(xg, add)[0]
    (out * w_rand).sum().backward()
    # oracle with the bf16-rounded weights and input the kernels actually consumed
    sd = {k: v.to(torch.bfloat16).float() for k, v in enc.state_dict().items()}
    o_out, o_dx, o_g = _oracle_run(sd, x.to(torch.bfloat16).float(), add, L, heads, w_rand)
    e_out, e_dx = rel(out, o_out), rel(xg.grad, o_dx)
    print("B%d S%d H%d L%d: out %.2e dx %.2e" % (B, S, H, L, e_out, e_dx))
    # measured (profiles/r2_parity_errors.txt): L=1 out 3.4e-3 / dx 3.8e-3 / worst dW 5.3e-3; L=2 4.8e-3 / 5.2e-3 / 7.5e-3
    assert e_out < 1e-2 and e_dx < 1e-2
    worst, worst_n = check_param_grads(enc.named_parameters(), o_g, 1e-2 if L == 1 else 1.5e-2)
    print("   worst dW %.2e (%s)" % (worst, worst_n))


def test_encoder_dropout_matches_oracle_with_same_masks():
    """train mode: run with p=0.1, pull the keep-bits the kernels generated, feed the same masks to the oracle"""
    from mmf_b200 import engine as E, functional as F
    from mmf_b200.modules import B200BertEncoder, EncoderRunner
    torch.manual_seed(3)
    B, S, H, heads, I = 2, 100, 128, 2, 256
    enc = B200BertEncoder(bert_cfg(H, heads, I, 1, p=0.1)).cuda().train()
    x = torch.randn(B, S, H, device="cuda")
    add = O.extended_attention_mask(torch.ones(B, S, dtype=torch.long, device="cuda"))
    captured = []
    orig = E.DropoutState.bits

    def spy(self, rows_shape, ncols, p, device):
        out = orig(self, rows_shape, ncols, p, device)
        captured.append((tuple(rows_shape), ncols, out))
        return out
    E.DropoutState.bits = spy
    try:
        xg = x.clone().requires_grad_(True)
        out = enc(xg, add)[0]
        w_rand = torch.randn_like(out)
        (out * w_rand).sum().backward()
    finally:
        E.DropoutState.bits = orig
    assert len(captured) == 3   # attention probs, self-output, output
    attn = F.unpack_keep_bits(captured[0][2], S)                       # [B,h,S,S]
    so = F.unpack_keep_bits(captured[1][2], H).view(B, S, H)
    oo = F.unpack_keep_bits(captured[2][2], H).view(B, S, H)
    for m in (attn, so, oo):
        frac = m.float().mean().item()
        assert 0.88 < frac < 0.92, frac                                 # P(keep) = 0.9
    sd = {k: v.to(torch.bfloat16).float() for k, v in enc.state_dict().items()}
    masks = [{"attn": attn, "self_out": so, "out": oo}]
    o_out, o_dx, o_g = _oracle_run(sd, x.to(torch.bfloat16).float(), add, 1, heads, w_rand, masks, 0.1)
    e_out, e_dx = rel(out, o_out), rel(xg.grad, o_dx)
    print("dropout parity: out %.2e dx %.2e" % (e_out, e_dx))
    assert e_out < 1e-2 and e_dx < 1e-2            # measured 3.1e-3 / 3.7e-3
    check_param_grads(enc.named_parameters(), o_g, 1.5e-2)


def test_grad_accumulation_and_zero_grad():
    """second backward accumulates in place into the flat gradient buffer; zero_grad(set_to_none) resets"""
    from mmf_b200.modules import B200BertEncoder
    torch.manual_seed(0)
    enc = B200BertEncoder(bert_cfg(128, 2, 256, 1)).cuda().eval()
    x = torch.randn(2, 40, 128, device="cuda")
    w = torch.randn(2, 40, 128, device="cuda")
    (enc(x)[0] * w).sum().backward()
    g1 = {n: p.grad.clone() for n, p in enc.named_parameters()}
    pack = enc._runner.pack
    p0 = next(enc.parameters())
    assert p0.grad.data_ptr() == pack.grad_view(p0).data_ptr()   # autograd installed the flat-buffer view, no copy
    (enc(x)[0] * w).sum().backward()
    for n, p in enc.named_parameters():
        assert rel(p.grad, 2 * g1[n]) < 1e-3, n
    enc.zero_grad(set_to_none=True)
    (enc(x)[0] * w).sum().backward()
    for n, p in enc.named_parameters():
        assert rel(p.grad, g1[n]) < 1e-3, n


def test_cpu_input_raises():
    from mmf_b200.modules import B200BertEncoder
    enc = B200BertEncoder(bert_cfg(128, 2, 256, 1))
    with pytest.raises(RuntimeError):
        enc(torch.zeros(1, 4, 128))


def test_vilbert_encoder_real_widths_vs_oracle():
    """BASELINE config 3 widths: text 768/12h/3072, image 1024/8h/1024, co-attention 1024/8h (d=128), T=R=36;
    a short schedule (2 text, 1 image, 1 connection layer) keeps the oracle fast."""
    from mmf_b200.modules import B200ViLBertEncoder
    torch.manual_seed(0)
    c = dict(hidden_size=768, num_attention_heads=12, intermediate_size=3072, num_hidden_layers=2,
             v_hidden_size=1024, v_num_attention_heads=8, v_intermediate_size=1024, v_num_hidden_layers=1,
             bi_hidden_size=1024, bi_num_attention_heads=8, v_biattention_id=[0], t_biattention_id=[1])
    cfg = types.SimpleNamespace(hidden_dropout_prob=0.0, v_hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                                v_attention_probs_dropout_prob=0.0, **c)
    enc = B200ViLBertEncoder(cfg).cuda().eval()
    with torch.no_grad():
        for n, p in enc.named_parameters():
            if p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.02)
    B, T, R = 4, 36, 36
    g = torch.Generator(device="cuda").manual_seed(1)
    txt = torch.randn(B, T, 768, generator=g, device="cuda")
    img = torch.randn(B, R, 1024, generator=g, device="cuda")
    tmask = (torch.arange(T, device="cuda")[None] < torch.tensor([36, 20, 30, 9], device="cuda")[:, None]).long()
    imask = (torch.arange(R, device="cuda")[None] < torch.tensor([36, 36, 12, 25], device="cuda")[:, None]).long()
    tadd, iadd = O.extended_attention_mask(tmask), O.extended_attention_mask(imask)
    wt = torch.randn(B, T, 768, generator=g, device="cuda")
    wv = torch.randn(B, R, 1024, generator=g, device="cuda")
    tg, ig = txt.clone().requires_grad_(True), img.clone().requires_grad_(True)
    tl, vl, _ = enc(tg, ig, tadd, tadd, iadd, None, output_all_encoded_layers=False)
    ((tl[-1] * wt).sum() + (vl[-1] * wv).sum()).backward()
    sd = {k: v.detach().to(torch.bfloat16).float().requires_grad_(True) for k, v in enc.state_dict().items()}
    tf = txt.to(torch.bfloat16).float().requires_grad_(True)
    vf = img.to(torch.bfloat16).float().requires_grad_(True)
    to, vo = O.vilbert_encoder(tf, vf, tadd, iadd, sd, "", c)
    ((to * wt).sum() + (vo * wv).sum()).backward()
    errs = {"t_out": rel(tl[-1], to), "v_out": rel(vl[-1], vo), "dtxt": rel(tg.grad, tf.grad), "dimg": rel(ig.grad, vf.grad)}
    print("vilbert real widths:", " ".join("%s=%.2e" % kv for kv in errs.items()))
    assert max(errs.values()) < 1.5e-2
    ref = {k: v.grad for k, v in sd.items() if v.grad is not None}
    unused = [n for n, p in enc.named_parameters() if n not in ref]
    assert all("q_dense" in n for n in unused)
    worst, wn = check_param_grads(enc.named_parameters(), ref, 2e-2, skip=unused)
    print("   worst dW %.2e (%s)" % (worst, wn))
    # train mode with the reference's dropout probabilities runs and stays finite
    enc.train()
    for m in enc.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.1
    tl, vl, _ = enc(txt, img, tadd, tadd, iadd, None)
    assert torch.isfinite(tl[-1]).all() and torch.isfinite(vl[-1]).all()


def test_bert_encoder_mmft_sequence_length():
    """BASELINE config 4: 128 text + 196 patch tokens = 324 -> three 128-row query tiles, 384 padded key columns"""
    from mmf_b200.modules import B200BertEncoder
    torch.manual_seed(0)
    B, S, H, heads, I = 2, 324, 768, 12, 3072
    enc = B200BertEncoder(bert_cfg(H, heads, I, 1)).cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.randn(B, S, H, generator=g, device="cuda")
    mask = torch.ones(B, S, dtype=torch.long, device="cuda")
    mask[1, 300:] = 0
    add = O.extended_attention_mask(mask)
    w_rand = torch.randn(B, S, H, generator=g, device="cuda")
    xg = x.clone().requires_grad_(True)
    out = enc(xg, add)[0]
    (out * w_rand).sum().backward()
    sd = {k: v.to(torch.bfloat16).float() for k, v in enc.state_dict().items()}
    o_out, o_dx, o_g = _oracle_run(sd, x.to(torch.bfloat16).float(), add, 1, heads, w_rand)
    e_out, e_dx = rel(out, o_out), rel(xg.grad, o_dx)
    print("S=324: out %.2e dx %.2e" % (e_out, e_dx))
    assert e_out < 1e-2 and e_dx < 1.5e-2
    check_param_grads(enc.named_parameters(), o_g, 2e-2)
