"""Embedding front-end (K1) + VisualBERT trunk on the GPU: reference goldens, oracle gradients, integer paths."""
import types

import pytest
import torch

from oracle import fusion_oracle as O
from oracle import golden_io

pytestmark = pytest.mark.gpu


def rel(a, b, floor=1e-3):
    fl = floor * (b.numel() ** 0.5)
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm().clamp_min(fl)).item()


def emb_cfg(H=64, V=50, P=32, F=40, p=0.0):
    return types.SimpleNamespace(hidden_size=H, vocab_size=V, max_position_embeddings=P, type_vocab_size=2,
                                 visual_embedding_dim=F, hidden_dropout_prob=p, layer_norm_eps=1e-12)


def test_visio_linguistic_embeddings_vs_reference_golden():
    from mmf_b200.embeddings import B200VisioLinguisticEmbeddings
    g = golden_io.load("embeddings")
    mod = B200VisioLinguisticEmbeddings(emb_cfg())
    assert set(mod.state_dict().keys()) == set(g["vl_state_dict"].keys())
    mod.load_state_dict(g["vl_state_dict"])
    mod = mod.cuda().eval()
    ids, seg, feats, vtype = (g[k].cuda() for k in ("ids", "seg", "feats", "vtype"))
    out = mod(ids, seg, feats, vtype)
    e1 = rel(out, g["out_plain"])
    out_t = mod(ids, seg)
    e2 = rel(out_t, g["out_text"])
    print("embeddings vs golden: text+image %.2e text-only %.2e" % (e1, e2))
    assert e1 < 1e-2 and e2 < 1e-2
    # image_text_alignment: position of a region = mean of its aligned words' position embeddings (+ pos_visual[0]);
    # one region of the fixture is aligned to nothing (divide-by-zero guard, embeddings.py:396-399)
    out_a = mod(ids, seg, feats, vtype, g["alignment"].cuda())
    e3 = rel(out_a, g["out_alignment"])
    print("embeddings with image_text_alignment vs golden: %.2e" % e3)
    assert e3 < 1e-2
    mod.zero_grad()
    mod.train()
    x = mod(ids, seg, feats, vtype, g["alignment"].cuda())
    (x.float() ** 2).sum().backward()
    assert mod.position_embeddings.weight.grad is not None and torch.isfinite(mod.position_embeddings.weight.grad).all()


def test_embeddings_backward_vs_oracle():
    from mmf_b200.embeddings import B200VisioLinguisticEmbeddings
    torch.manual_seed(1)
    H, V, P, Fd, B, T, R = 128, 200, 64, 256, 3, 20, 12
    mod = B200VisioLinguisticEmbeddings(emb_cfg(H, V, P, Fd)).cuda().eval()
    with torch.no_grad():
        mod.LayerNorm.weight.add_(torch.randn(H, device="cuda") * 0.05)
        mod.projection.bias.add_(torch.randn(H, device="cuda") * 0.05)
    ids = torch.randint(0, V, (B, T), device="cuda")
    ids[:, 3] = ids[:, 2]                      # repeated token -> accumulating scatter
    seg = torch.randint(0, 2, (B, T), device="cuda")
    feats = torch.randn(B, R, Fd, device="cuda").abs().requires_grad_(True)
    vtype = torch.zeros(B, R, dtype=torch.long, device="cuda")
    w = torch.randn(B, T + R, H, device="cuda")
    out = mod(ids, seg, feats, vtype)
    (out * w).sum().backward()
    sd = {"e." + k: v.detach().to(torch.bfloat16).float().requires_grad_(True) for k, v in mod.state_dict().items()}
    fr = feats.detach().to(torch.bfloat16).float().requires_grad_(True)
    ref = O.visio_linguistic_embeddings(ids, seg, fr, vtype, sd, "e")
    (ref * w).sum().backward()
    assert rel(out, ref) < 1e-2
    assert rel(feats.grad, fr.grad) < 1.5e-2
    worst = 0.0
    for n, p in mod.named_parameters():
        e = rel(p.grad, sd["e." + n].grad)
        worst = max(worst, e)
        assert e < 2e-2, (n, e)
    print("embedding grads vs oracle: worst %.2e" % worst)


def test_visual_bert_sample_list_path_and_integer_masks():
    from mmf_b200.visual_bert import B200VisualBERT, image_mask_from_dims
    torch.manual_seed(2)
    cfg = types.SimpleNamespace(hidden_size=128, num_attention_heads=2, intermediate_size=256, num_hidden_layers=2,
                                vocab_size=100, max_position_embeddings=64, type_vocab_size=2, visual_embedding_dim=64,
                                hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, layer_norm_eps=1e-12)
    model = B200VisualBERT(cfg).cuda().eval()
    B, T, R = 3, 16, 10
    maxf = torch.tensor([10, 4, 7], device="cuda")
    lens = [16, 9, 12]
    mask = torch.zeros(B, T, dtype=torch.long, device="cuda")
    for b, n in enumerate(lens):
        mask[b, :n] = 1
    sl = {"input_ids": torch.randint(0, 100, (B, T), device="cuda"), "input_mask": mask,
          "segment_ids": torch.zeros(B, T, dtype=torch.long, device="cuda"),
          "image_feature_0": torch.randn(B, R, 64, device="cuda").abs(), "image_info_0": {"max_features": maxf}}
    out = model(sl)
    im, vtype, att = O.visual_bert_masks(mask, maxf, R)
    assert torch.equal(out["image_mask"], im)                      # bit-exact integer paths
    assert torch.equal(out["attention_mask"], att)
    assert torch.equal(image_mask_from_dims(maxf, R), im)
    sd = {k: v.detach().to(torch.bfloat16).float() for k, v in model.state_dict().items()}
    emb = O.visio_linguistic_embeddings(sl["input_ids"], sl["segment_ids"], sl["image_feature_0"].to(torch.bfloat16).float(),
                                        vtype, sd, "bert.embeddings")
    seq = O.bert_encoder(emb, O.extended_attention_mask(att), sd, "bert.encoder", 2, 2)
    pooled = O.bert_pooler(seq, sd, "bert.pooler")
    assert rel(out["sequence_output"], seq) < 1e-2
    assert rel(out["pooled_output"], pooled) < 1e-2
