"""SURVEY.md 8a row a13 on the GPU: the ReLU GEMM epilogue + its backward, the fc7 region-feature encoder and the
TransformerEncoder wrapper against the reference's own outputs (tests/golden/encoders.*.pt), incl. the padding_idx
rule of HF word embeddings (the [PAD] row is read but gets no gradient)."""

import pytest
import torch

from oracle import golden_io

pytestmark = pytest.mark.gpu


def rel(a, b, floor=1e-3):
    fl = floor * (b.numel() ** 0.5)
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm().clamp_min(fl)).item()


def gold():
    return golden_io.load("encoders")


@pytest.mark.parametrize("M,N,K", [(300, 128, 256), (1000, 2048, 2048), (77, 264, 72)])
def test_relu_epilogue_and_backward(M, N, K):
    from mmf_b200 import functional as F, lib
    torch.manual_seed(M)
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda") / K ** 0.5).to(torch.bfloat16)
    b = torch.randn(N, device="cuda").to(torch.bfloat16)
    y = F.gemm(x, w, epi=lib.EPI_BIAS_RELU, bias=b)
    ref = torch.relu(x.float() @ w.float().t() + b.float())
    assert (y >= 0).all()
    assert rel(y, ref) < 1e-2
    dy = torch.randn(M, N, device="cuda").to(torch.bfloat16)
    dz = F.relu_bwd(dy, y)
    assert torch.equal(dz, torch.where(y > 0, dy, torch.zeros_like(dy)))      # selection only: bit-exact


def test_relu_bwd_ragged_tail_and_errors():
    from mmf_b200 import functional as F
    y = torch.randn(3, 13, device="cuda").to(torch.bfloat16)      # 39 elements: scalar tail path
    dy = torch.randn(3, 13, device="cuda").to(torch.bfloat16)
    assert torch.equal(F.relu_bwd(dy, y), torch.where(y > 0, dy, torch.zeros_like(dy)))
    with pytest.raises(ValueError):
        F.relu_bwd(dy, y[:2])


def test_fc7_encoder_vs_reference_golden():
    from mmf_b200.encoders import B200FinetuneFasterRcnnFpnFc7
    f = gold()["fc7"]
    enc = B200FinetuneFasterRcnnFpnFc7({"in_dim": 256, "out_dim": 128})
    # checkpoints written before the `module.` prefix was dropped still load (encoders.py:151-174)
    enc.load_state_dict({"module." + k: v for k, v in f["state_dict"].items()})
    enc = enc.cuda()
    x = f["feat"].cuda().requires_grad_(True)
    y = enc(x)
    assert y.shape == f["out"].shape and y.dtype == x.dtype
    assert rel(y, f["out"]) < 1e-2
    wr = f["w_rand"].cuda()
    (y * wr).sum().backward()
    # ReLU is discontinuous: a pre-activation within bf16 rounding of 0 may land on the other side of the kink, and
    # that element's whole gradient then differs from the fp32 reference.  So (i) the kept/dropped pattern must agree
    # with the reference except where the reference pre-activation is tiny, and (ii) the gradients must match the
    # reference formulas evaluated with the pattern the GPU actually used.
    W, bias = f["state_dict"]["lc.weight"].cuda(), f["state_dict"]["lc.bias"].cuda()
    pre = f["feat"].cuda() @ W.t() + bias
    flips = (y > 0) != (f["out"].cuda() > 0)
    assert flips.float().mean() < 0.01 and (pre[flips].abs() < 0.05).all()
    dz = wr * (y > 0)
    assert rel(x.grad, dz @ W) < 1e-2
    assert rel(enc.lc.weight.grad, dz.reshape(-1, 128).t() @ f["feat"].cuda().reshape(-1, 256)) < 1e-2
    assert rel(enc.lc.bias.grad, dz.reshape(-1, 128).sum(0)) < 1e-2
    # and against the reference's own gradients with a tolerance that covers the flipped elements
    assert rel(x.grad, f["dfeat"]) < 6e-2 and rel(enc.lc.weight.grad, f["grads"]["lc.weight"]) < 6e-2
    with pytest.raises(RuntimeError):
        B200FinetuneFasterRcnnFpnFc7({"in_dim": 256, "out_dim": 128})(f["feat"])      # CPU tensor: no fallback


def test_transformer_encoder_vs_reference_golden():
    from mmf_b200.encoders import B200TransformerEncoder
    t = gold()["transformer"]
    c = t["cfg"]
    te = B200TransformerEncoder(dict(hidden_size=c["hidden"], num_hidden_layers=c["layers"],
                                     num_attention_heads=c["heads"], intermediate_size=c["inter"], vocab_size=c["vocab"],
                                     max_position_embeddings=c["max_pos"], num_segments=c["num_segments"]))
    assert te.embeddings.token_type_embeddings.weight.shape[0] == c["num_segments"]
    w = te.embeddings.token_type_embeddings.weight
    assert torch.equal(w[2], w[3])                    # rows 2..n-2 start at the mean of the two pretrained rows
    te.load_state_dict(t["state_dict"])
    te = te.cuda().eval()
    ids, mask, seg = t["ids"].cuda(), t["mask"].cuda(), t["seg"].cuda()
    assert (ids == 0).any()                          # the fixture exercises the [PAD] row
    pooled = te(ids, mask, seg)
    seq = te(ids, mask, seg, return_sequence=True)
    e1, e2 = rel(seq, t["seq"]), rel(pooled, t["pooled"])
    print("transformer encoder vs golden: seq %.2e pooled %.2e" % (e1, e2))
    assert e1 < 1e-2 and e2 < 1e-2
    ((seq * t["w_seq"].cuda()).sum() + (pooled * t["w_pooled"].cuda()).sum()).backward()
    named = dict(te.named_parameters())
    # the reference arithmetic itself in bf16 (oracle with bf16 weights) against its fp32 golden: the per-parameter
    # drift that bounds what any bf16 implementation can reach on this 12-token fixture (see test_encoder_gpu.py)
    from oracle import fusion_oracle as O
    sdb = {k: v.cuda().to(torch.bfloat16).requires_grad_(True) for k, v in t["state_dict"].items()
           if k.startswith("module.")}
    oseq = O.transformer_encoder(ids, mask, seg, sdb, "module", c["layers"], c["heads"], True)
    opool = O.transformer_encoder(ids, mask, seg, sdb, "module", c["layers"], c["heads"])
    ((oseq.float() * t["w_seq"].cuda()).sum() + (opool.float() * t["w_pooled"].cuda()).sum()).backward()
    drift = {k: rel(v.grad, t["grads"][k]) for k, v in sdb.items() if v.grad is not None}
    errs, bad = {}, []
    for k, p in named.items():
        if p.grad is None:
            continue
        if ".key.bias" in k:      # analytically zero (softmax is shift invariant): only required to be tiny
            assert p.grad.float().norm() <= 0.05 * named[k.replace("key", "query")].grad.float().norm() + 1e-3, k
            continue
        errs[k] = rel(p.grad, t["grads"][k])
        if errs[k] >= max(2e-2, 2.5 * drift.get(k, 0.0)):
            bad.append((k, "%.2e" % errs[k], "%.2e" % drift.get(k, 0.0)))
    wk = max(errs, key=errs.get)
    print("worst gradient error %.2e (%s), bf16-reference drift there %.2e" % (errs[wk], wk, drift.get(wk, 0.0)))
    assert not bad, bad[:8]
    gw = named["module.embeddings.word_embeddings.weight"].grad
    assert torch.count_nonzero(gw[0]) == 0            # padding_idx row: no gradient, as in the reference
    assert torch.count_nonzero(t["grads"]["module.embeddings.word_embeddings.weight"][0]) == 0


def test_visio_linguistic_embeddings_padding_row_gets_no_gradient():
    import types
    from mmf_b200.embeddings import B200VisioLinguisticEmbeddings
    cfg = types.SimpleNamespace(hidden_size=128, vocab_size=50, max_position_embeddings=64, type_vocab_size=2,
                                hidden_dropout_prob=0.0, visual_embedding_dim=64, layer_norm_eps=1e-12,
                                initializer_range=0.02)
    emb = B200VisioLinguisticEmbeddings(cfg).cuda()
    ids = torch.tensor([[5, 7, 0, 0], [9, 0, 3, 0]], device="cuda")
    feats = torch.randn(2, 3, 64, device="cuda")
    out = emb(ids, torch.zeros_like(ids), feats, torch.zeros(2, 3, dtype=torch.long, device="cuda"))
    out.float().square().sum().backward()
    g = emb.word_embeddings.weight.grad
    assert torch.count_nonzero(g[0]) == 0 and torch.count_nonzero(g[5]) > 0 and torch.count_nonzero(g[3]) > 0
