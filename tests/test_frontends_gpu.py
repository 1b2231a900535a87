"""MMBT, MMFTransformer backend, ViLBERT image embeddings and the monkey-patch swap on the GPU, against the
reference's own outputs (tests/golden) and oracle gradients."""
import types

import pytest
import torch

from oracle import fusion_oracle as O
from oracle import golden_io

pytestmark = pytest.mark.gpu


def rel(a, b, floor=1e-3):
    fl = floor * (b.numel() ** 0.5)
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm().clamp_min(fl)).item()


def bert_cfg(hidden, heads, inter, layers, **kw):
    d = dict(hidden_size=hidden, num_attention_heads=heads, intermediate_size=inter, num_hidden_layers=layers,
             hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, layer_norm_eps=1e-12, hidden_act="gelu",
             initializer_range=0.02, vocab_size=50, max_position_embeddings=64, type_vocab_size=2)
    d.update(kw)
    return types.SimpleNamespace(**d)


def test_mmbt_vs_reference_golden_and_integer_paths():
    from mmf_b200.mmbt import B200MMBTBase
    g = golden_io.load("mmbt")
    c = g["cfg"]
    base = B200MMBTBase(bert_cfg(c["hidden"], c["heads"], c["inter"], c["layers"], modal_hidden_size=c["modal_hidden"]))
    sd = base.mmbt.state_dict()
    assert set(g["state_dict"].keys()) <= set(sd.keys())          # reference keys (incl. the shared modal_encoder.* aliases)
    base.mmbt.load_state_dict(g["state_dict"], strict=False)
    base = base.cuda().eval()
    sl = {"input_ids": g["ids"].cuda().clone(), "input_mask": g["mask"].cuda().clone(), "segment_ids": g["seg"].cuda(),
          "image_feature_0": g["feats"].cuda()}
    seq, pooled, _ = base(sl)
    # integer token surgery is bit-exact with the reference (tests/models/test_mmbt.py:68-103 in the reference)
    assert torch.equal(sl["input_ids"].cpu(), g["shifted_ids"])
    assert torch.equal(sl["input_mask"].cpu(), g["shifted_mask"])
    e1, e2 = rel(seq, g["seq_out"]), rel(pooled, g["pooled"])
    print("mmbt vs golden: seq %.2e pooled %.2e" % (e1, e2))
    assert e1 < 1e-2 and e2 < 1e-2


def test_mmbt_with_fc7_modal_encoder_built_from_config():
    # configs/models/mmbt/with_features.yaml: region features -> fc7 relu(Linear) -> MMBT, built the reference's way
    from mmf_b200.mmbt import B200MMBTBase
    torch.manual_seed(3)
    cfg = dict(direct_features_input=True, modal_hidden_size=128, num_labels=2,
               text_encoder=dict(type="transformer",
                                 params=dict(hidden_size=128, num_hidden_layers=1, num_attention_heads=2, vocab_size=50,
                                             max_position_embeddings=64, num_segments=2, hidden_dropout_prob=0.0,
                                             attention_probs_dropout_prob=0.0)),
               modal_encoder=dict(type="finetune_faster_rcnn_fpn_fc7", params=dict(in_dim=64, out_dim=128)))
    base = B200MMBTBase.from_config(cfg).cuda().eval()
    B, T, R = 2, 10, 7
    ids = torch.randint(3, 50, (B, T), device="cuda")
    mask = torch.ones(B, T, dtype=torch.long, device="cuda")
    mask[1, 6:] = 0
    seg = torch.zeros(B, T, dtype=torch.long, device="cuda")
    feats = torch.randn(B, R, 64, device="cuda")
    sl = {"input_ids": ids.clone(), "input_mask": mask.clone(), "segment_ids": seg, "image_feature_0": feats}
    seq, pooled, _ = base(sl)
    w = torch.randn_like(seq)
    (seq * w).sum().backward()
    sd = {k: v.detach().to(torch.bfloat16).float().requires_grad_(True) for k, v in base.mmbt.state_dict().items()}
    fc7 = O.fc7_encoder(feats.to(torch.bfloat16).float(), sd, "modal_encoder.encoder")
    oseq, opooled, _ = O.mmbt_forward(fc7, ids, mask, seg, sd, {"num_hidden_layers": 1, "num_attention_heads": 2})
    (oseq * w).sum().backward()
    assert rel(seq, oseq) < 1e-2 and rel(pooled, opooled) < 1e-2
    named = dict(base.mmbt.named_parameters())
    assert rel(named["modal_encoder.proj_embeddings.weight"].grad, sd["modal_encoder.proj_embeddings.weight"].grad) < 2e-2
    # the fc7 weight gradient crosses the ReLU kink: a few pre-activations flip side in bf16 (test_encoders_gpu.py)
    assert rel(named["modal_encoder.encoder.lc.weight"].grad, sd["modal_encoder.encoder.lc.weight"].grad) < 6e-2
    assert rel(named["modal_encoder.encoder.lc.bias"].grad, sd["modal_encoder.encoder.lc.bias"].grad) < 6e-2


def test_mmbt_backward_vs_oracle():
    from mmf_b200.mmbt import B200MMBTBase
    torch.manual_seed(0)
    cfg = bert_cfg(128, 2, 256, 1, modal_hidden_size=64, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    base = B200MMBTBase(cfg).cuda().eval()
    B, T, R = 2, 10, 7
    ids = torch.randint(3, 50, (B, T), device="cuda")
    mask = torch.ones(B, T, dtype=torch.long, device="cuda")
    mask[1, 6:] = 0
    seg = torch.zeros(B, T, dtype=torch.long, device="cuda")
    feats = torch.randn(B, R, 64, device="cuda").abs()
    sl = {"input_ids": ids.clone(), "input_mask": mask.clone(), "segment_ids": seg, "image_feature_0": feats}
    seq, pooled, _ = base(sl)
    w = torch.randn_like(seq)
    (seq * w).sum().backward()
    sd = {k: v.detach().to(torch.bfloat16).float().requires_grad_(True) for k, v in base.mmbt.state_dict().items()}
    oseq, _, _ = O.mmbt_forward(feats.to(torch.bfloat16).float(), ids, mask, seg, sd,
                                {"num_hidden_layers": 1, "num_attention_heads": 2})
    (oseq * w).sum().backward()
    assert rel(seq, oseq) < 1e-2
    named = dict(base.mmbt.named_parameters())
    for n in ("modal_encoder.proj_embeddings.weight", "transformer.embeddings.word_embeddings.weight",
              "transformer.embeddings.position_embeddings.weight", "transformer.embeddings.LayerNorm.weight",
              "transformer.encoder.layer.0.intermediate.dense.weight"):
        og = sd[n].grad
        if n.startswith("transformer.embeddings.") and ("modal_encoder." + n.split("embeddings.")[1]) in sd:
            alias = sd["modal_encoder." + n.split("embeddings.")[1]].grad   # shared tensor: oracle dict holds two copies
            if alias is not None:
                og = og + alias
        e = rel(named[n].grad, og)
        assert e < 2e-2, (n, e)


def test_mmft_backend_vs_reference_golden():
    from mmf_b200.mmft_backend import B200TransformerBackend
    from mmf_b200.registry import registry
    g = golden_io.load("mmft_embeddings")
    tcfg = bert_cfg(64, 1, 128, 1, max_position_embeddings=32, pad_token_id=0)
    mods = [dict(type="text", key="text", position_dim=32, embedding_dim=64, segment_id=0),
            dict(type="image", key="image", position_dim=16, embedding_dim=40, segment_id=1)]
    cfg = dict(modalities=mods, transformer_config=tcfg, token_noise_mean=0.0, token_noise_std=0.01)
    backend = registry.get_transformer_backend_class("b200")(cfg)
    assert set(backend.embeddings.state_dict().keys()) == set(g["state_dict"].keys())
    backend.embeddings.load_state_dict(g["state_dict"])
    backend = backend.cuda().eval()
    cu = lambda d: {k: v.cuda() for k, v in d.items()}
    emb = backend.generate_embeddings(cu(g["tokens"]), cu(g["pos"]), cu(g["seg"]), None)
    e = rel(emb, g["out"])
    print("mmft embeddings vs golden: %.2e" % e)
    assert e < 1e-2
    am = backend.generate_attention_mask([m.cuda() for m in g["masks"]])
    assert torch.equal(am.cpu(), g["attention_mask"])                      # mask construction is exact
    seq, first = backend(cu(g["tokens"]), cu(g["pos"]), cu(g["seg"]), [m.cuda() for m in g["masks"]])
    assert seq.shape == (2, 11, 64) and torch.isfinite(seq.float()).all()
    # weight tying surface used by MMFT heads (mmf_transformer.py:172-174)
    assert backend.embeddings.token_embeddings[0].weight is backend.transformer.embeddings.word_embeddings.weight


def test_vilbert_image_embeddings_vs_reference_golden():
    from mmf_b200.vilbert import B200ImageFeatureEmbeddings
    g = golden_io.load("embeddings")
    mod = B200ImageFeatureEmbeddings(types.SimpleNamespace(v_feature_size=40, v_hidden_size=96, hidden_dropout_prob=0.1))
    assert set(mod.state_dict().keys()) == set(g["img_state_dict"].keys())
    mod.load_state_dict(g["img_state_dict"])
    mod = mod.cuda().eval()
    feats = g["feats"].cuda().requires_grad_(True)
    out = mod(feats, g["loc"].cuda())
    e = rel(out, g["img_out"])
    print("vilbert image embeddings vs golden: %.2e" % e)
    assert e < 1e-2
    (out.float() ** 2).sum().backward()
    assert mod.image_location_embeddings.weight.grad is not None and feats.grad is not None


def test_monkey_patch_swap_on_hf_bert_encoder():
    """replace_with_b200(): a stock HuggingFace BertEncoder instance runs on the engine, parameters keep their names"""
    from transformers import BertConfig
    from transformers.models.bert.modeling_bert import BertEncoder
    from mmf_b200.patch import replace_with_b200, undo_replace_with_b200
    torch.manual_seed(0)
    cfg = BertConfig(hidden_size=128, num_attention_heads=2, intermediate_size=256, num_hidden_layers=2, vocab_size=50,
                     hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    enc = BertEncoder(cfg).cuda().eval()
    keys = set(enc.state_dict().keys())
    x = torch.randn(2, 20, 128, device="cuda")
    mask = torch.ones(2, 20, dtype=torch.long, device="cuda")
    mask[0, 15:] = 0
    add = O.extended_attention_mask(mask)
    orig_forward = BertEncoder.forward
    replace_with_b200()
    try:
        out = enc(x, add)[0]
    finally:
        undo_replace_with_b200()
    assert BertEncoder.forward is orig_forward
    assert set(enc.state_dict().keys()) == keys
    sd = {k: v.detach().to(torch.bfloat16).float() for k, v in enc.state_dict().items()}
    ref = O.bert_encoder(x.to(torch.bfloat16).float(), add, sd, "", 2, 2)
    assert rel(out, ref) < 1e-2
