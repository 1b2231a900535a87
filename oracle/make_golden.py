"""TEST INFRASTRUCTURE - generates tests/golden/*.pt by running the REFERENCE's own source files.

Runs only in the build container (needs /root/reference):   python -m oracle.make_golden
Each fixture holds seeded weights (reference state_dict key names), inputs, the reference's outputs
and the gradients of a fixed random-projection loss  (out * W_rand).sum()  (SURVEY.md 8d: out.sum()
is degenerate after a final LayerNorm).  Shapes are tiny; a fixture over 1 MB is stored in parts (oracle/golden_io.py).
All modules run in eval mode (dropout off): the reference's RNG stream is not reproducible elsewhere.
"""
import json
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import golden_io  # noqa: E402
from oracle import ref_loader as R  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def _perturb(module, seed):
    """reference init (normal 0.02, zero bias, LN 1/0) + small perturbation of biases / LN so they matter"""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in module.named_parameters():
            if p.dim() >= 2:
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            elif "LayerNorm.weight" in n or n.endswith("layer_norms.0.weight") or n.endswith(".1.weight"):
                p.copy_(1.0 + torch.randn(p.shape, generator=g) * 0.02)
            else:
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)


def _grads(module, names):
    sd = dict(module.named_parameters())
    return {n: sd[n].grad.detach().clone() for n in names if sd[n].grad is not None}


def _save(name, obj):
    for path in golden_io.save(name, obj, OUT):
        print("wrote %s (%.1f KB)" % (path, os.path.getsize(path) / 1024))


def golden_bert_encoder():
    from transformers import BertConfig
    hl = R.hf_layers()
    # head_dim 64 (the reference's 768/12): the fused attention kernel supports head_dim 64 and 128
    cfg = BertConfig(hidden_size=128, num_attention_heads=2, intermediate_size=256, num_hidden_layers=2,
                     vocab_size=50, max_position_embeddings=32)
    enc = hl.BertEncoderJit(cfg).eval()
    _perturb(enc, 11)
    g = torch.Generator().manual_seed(12)
    B, S = 3, 12
    x = torch.randn(B, S, 128, generator=g, requires_grad=True)
    mask = torch.ones(B, S, dtype=torch.long)
    mask[0, 9:] = 0
    mask[1, 5:] = 0
    mask[2, :] = 0  # fully masked row: softmax must become uniform, not NaN (tests/models/test_vilbert.py:66)
    add = (1.0 - mask[:, None, None, :].float()) * -10000.0
    out = enc(x, add)[0]
    w = torch.randn(out.shape, generator=g)
    (out * w).sum().backward()
    names = [n for n, _ in enc.named_parameters()]
    _save("bert_encoder", {
        "cfg": {"hidden": 128, "heads": 2, "inter": 256, "layers": 2},
        "state_dict": {k: v.detach().clone() for k, v in enc.state_dict().items()},
        "x": x.detach(), "mask": mask, "w_rand": w, "out": out.detach(), "dx": x.grad.detach(),
        "grads": _grads(enc, names),
    })


def golden_vilbert_encoder():
    vb = R.vilbert()
    cfg = types.SimpleNamespace(
        hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=3,
        v_hidden_size=128, v_num_attention_heads=1, v_intermediate_size=128, v_num_hidden_layers=2,
        bi_hidden_size=128, bi_num_attention_heads=2, v_biattention_id=[0, 1], t_biattention_id=[1, 2],
        hidden_act="gelu", v_hidden_act="gelu", hidden_dropout_prob=0.1, v_hidden_dropout_prob=0.1,
        attention_probs_dropout_prob=0.1, v_attention_probs_dropout_prob=0.1, layer_norm_eps=1e-12,
        fast_mode=False, with_coattention=True, in_batch_pairs=False, fixed_t_layer=0, fixed_v_layer=0,
        dynamic_attention=False, visualization=False, chunk_size_feed_forward=0, is_decoder=False,
        add_cross_attention=False, position_embedding_type="absolute", _attn_implementation="eager",
    )
    enc = vb.BertEncoder(cfg).eval()
    _perturb(enc, 21)
    g = torch.Generator().manual_seed(22)
    B, T, Rn = 2, 7, 5
    txt = torch.randn(B, T, 64, generator=g, requires_grad=True)
    img = torch.randn(B, Rn, 128, generator=g, requires_grad=True)
    tmask = torch.ones(B, T, dtype=torch.long)
    tmask[1, 4:] = 0
    imask = torch.ones(B, Rn, dtype=torch.long)
    imask[0, 3:] = 0
    tadd = (1.0 - tmask[:, None, None, :].float()) * -10000.0
    iadd = (1.0 - imask[:, None, None, :].float()) * -10000.0
    co = torch.zeros(B, 1, Rn, T)
    t_layers, v_layers, _ = enc(txt, img, tadd, tadd, iadd, co, output_all_encoded_layers=False)
    t_out, v_out = t_layers[-1], v_layers[-1]
    wt = torch.randn(t_out.shape, generator=g)
    wv = torch.randn(v_out.shape, generator=g)
    ((t_out * wt).sum() + (v_out * wv).sum()).backward()
    names = [n for n, p in enc.named_parameters()]
    grads = _grads(enc, names)
    unused = [n for n, p in enc.named_parameters() if p.grad is None]
    _save("vilbert_encoder", {
        "cfg": {k: getattr(cfg, k) for k in ("hidden_size", "num_attention_heads", "intermediate_size",
                                              "num_hidden_layers", "v_hidden_size", "v_num_attention_heads",
                                              "v_intermediate_size", "v_num_hidden_layers", "bi_hidden_size",
                                              "bi_num_attention_heads", "v_biattention_id", "t_biattention_id")},
        "state_dict": {k: v.detach().clone() for k, v in enc.state_dict().items()},
        "txt": txt.detach(), "img": img.detach(), "tmask": tmask, "imask": imask, "wt": wt, "wv": wv,
        "t_out": t_out.detach(), "v_out": v_out.detach(), "dtxt": txt.grad.detach(), "dimg": img.grad.detach(),
        "grads": grads, "unused": unused,
    })


def golden_embeddings():
    from transformers import BertConfig
    em = R.embeddings()
    vb = R.vilbert()
    cfg = BertConfig(hidden_size=64, vocab_size=50, max_position_embeddings=32, type_vocab_size=2)
    cfg.visual_embedding_dim = 40
    mod = em.BertVisioLinguisticEmbeddings(cfg).eval()
    _perturb(mod, 31)
    g = torch.Generator().manual_seed(32)
    B, T, Rn = 2, 9, 6
    ids = torch.randint(0, 50, (B, T), generator=g)
    seg = torch.randint(0, 2, (B, T), generator=g)
    feats = torch.randn(B, Rn, 40, generator=g).abs()
    vtype = torch.zeros(B, Rn, dtype=torch.long)
    out_plain = mod(ids, seg, feats, vtype)
    ali = torch.randint(-1, T, (B, Rn, 3), generator=g)
    ali[0, 0, :] = -1  # a region aligned to nothing: the divide-by-zero guard
    out_ali = mod(ids, seg, feats, vtype, ali)
    out_text = mod(ids, seg)
    # ViLBERT image embeddings
    vcfg = types.SimpleNamespace(v_feature_size=40, v_hidden_size=96, hidden_dropout_prob=0.1)
    imod = vb.BertImageFeatureEmbeddings(vcfg).eval()
    _perturb(imod, 33)
    loc = torch.rand(B, Rn, 5, generator=g)
    iout = imod(feats, loc)
    _save("embeddings", {
        "vl_state_dict": {k: v.detach().clone() for k, v in mod.state_dict().items() if v.dtype.is_floating_point},
        "ids": ids, "seg": seg, "feats": feats, "vtype": vtype, "alignment": ali,
        "out_plain": out_plain.detach(), "out_alignment": out_ali.detach(), "out_text": out_text.detach(),
        "img_state_dict": {k: v.detach().clone() for k, v in imod.state_dict().items()},
        "loc": loc, "img_out": iout.detach(),
    })


def golden_mmbt():
    from transformers import BertConfig
    hl = R.hf_layers()
    mm = R.mmbt()
    hl.replace_with_jit = lambda: None
    cfg = BertConfig(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=1,
                     vocab_size=50, max_position_embeddings=64, type_vocab_size=2)
    cfg.modal_hidden_size = 40
    transformer = hl.BertModelJit(cfg)
    model = mm.MMBTModel(cfg, transformer, torch.nn.Identity()).eval()
    _perturb(model, 41)
    g = torch.Generator().manual_seed(42)
    B, T, Rn = 2, 8, 10
    ids = torch.randint(3, 50, (B, T), generator=g)
    ids[:, 0] = 1  # [CLS]
    lens = [8, 5]
    mask = torch.zeros(B, T, dtype=torch.long)
    for b, n in enumerate(lens):
        mask[b, :n] = 1
        ids[b, n - 1] = 2  # [SEP]
    seg = torch.zeros(B, T, dtype=torch.long)
    feats = torch.randn(B, Rn, 40, generator=g).abs()
    # integer token surgery of MMBTBase.forward / extract_modal_end_token (bit-exact path)
    sl = {"input_ids": ids.clone(), "input_mask": mask.clone(), "segment_ids": seg.clone()}
    start = sl["input_ids"][:, 0].clone()
    end = mm.MMBTBase.extract_modal_end_token(None, sl)
    modal_tt = torch.full((B, 1), 1, dtype=torch.long)  # single segment, max_id == 0 -> token_value 1
    out = model(feats, input_ids=sl["input_ids"], modal_start_tokens=start, modal_end_tokens=end,
                attention_mask=sl["input_mask"], token_type_ids=sl["segment_ids"], modal_token_type_ids=modal_tt)
    _save("mmbt", {
        "cfg": {"hidden": 64, "heads": 1, "inter": 128, "layers": 1, "modal_hidden": 40},
        "state_dict": {k: v.detach().clone() for k, v in model.state_dict().items() if v.dtype.is_floating_point},
        "ids": ids, "mask": mask, "seg": seg, "feats": feats,
        "end_token": end, "shifted_ids": sl["input_ids"], "shifted_mask": sl["input_mask"],
        "seq_out": out[0].detach(), "pooled": out[1].detach(),
    })


class _Cfg(dict):
    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)


def golden_mmft_embeddings():
    from transformers import BertConfig
    hl = R.hf_layers()
    hb = R.hf_backend()
    tcfg = BertConfig(hidden_size=64, num_attention_heads=4, intermediate_size=128, num_hidden_layers=1,
                      vocab_size=50, max_position_embeddings=32, type_vocab_size=2, pad_token_id=0)
    transformer = hl.BertModelJit(tcfg)
    mcfg = _Cfg(modalities=[_Cfg(type="text", key="text", position_dim=32, embedding_dim=64, segment_id=0),
                            _Cfg(type="image", key="image", position_dim=16, embedding_dim=40, segment_id=1)],
                token_noise_mean=0.0, token_noise_std=0.01)
    torch.manual_seed(51)
    emb = hb.HuggingfaceEmbeddings(mcfg, tcfg, transformer).eval()
    _perturb(emb, 52)
    g = torch.Generator().manual_seed(53)
    B, T, P = 2, 7, 4
    tokens = {"text": torch.randint(0, 50, (B, T), generator=g), "image": torch.randn(B, P, 40, generator=g)}
    pos = {"text": torch.arange(T).unsqueeze(0).expand(B, T).contiguous(),
           "image": torch.arange(P).unsqueeze(0).expand(B, P).contiguous()}
    seg = {"text": torch.zeros(B, T, dtype=torch.long), "image": torch.ones(B, P, dtype=torch.long)}
    out = emb(tokens, pos, seg)
    masks = [torch.ones(B, T), torch.ones(B, P)]
    masks[0][1, 5:] = 0
    am = hb.HuggingfaceBackend.generate_attention_mask(None, masks)
    _save("mmft_embeddings", {
        "state_dict": {k: v.detach().clone() for k, v in emb.state_dict().items()},
        "tokens": tokens, "pos": pos, "seg": seg, "out": out.detach(), "masks": masks, "attention_mask": am,
    })


def golden_encoders():
    """encoders.py row a13: fc7 relu(Linear) and TransformerEncoder (BertModelJit + widened segment table).
    Both constructors read the network / pickles, so the objects are assembled around the reference's own
    `forward` / `_init_segment_embeddings` (the code under test) without running `__init__`."""
    from transformers import BertConfig
    enc = R.encoders()
    hl = R.hf_layers()
    g = torch.Generator().manual_seed(61)
    # --- FinetuneFasterRcnnFpnFc7.forward (encoders.py:176-179)
    fc7 = enc.FinetuneFasterRcnnFpnFc7.__new__(enc.FinetuneFasterRcnnFpnFc7)
    torch.nn.Module.__init__(fc7)
    fc7.lc = torch.nn.Linear(256, 128)
    fc7.out_dim = 128
    _perturb(fc7, 62)
    feat = torch.randn(3, 10, 256, generator=g, requires_grad=True)
    y = fc7(feat)
    wy = torch.randn(y.shape, generator=g)
    (y * wy).sum().backward()
    # legacy `module.` prefix handling (encoders.py:151-174)
    legacy = {"module.lc.weight": fc7.lc.weight.detach().clone(), "module.lc.bias": fc7.lc.bias.detach().clone()}
    fc7.load_state_dict(dict(legacy))
    # --- TransformerEncoder: BertModelJit (hf_layers.py:358-475) + _init_segment_embeddings (encoders.py:563-575)
    cfg = BertConfig(hidden_size=128, num_attention_heads=2, intermediate_size=256, num_hidden_layers=2,
                     vocab_size=50, max_position_embeddings=32)
    te = enc.TransformerEncoder.__new__(enc.TransformerEncoder)
    torch.nn.Module.__init__(te)
    te.module = hl.BertModelJit(cfg)
    _perturb(te.module, 63)
    pre_types = te.module.embeddings.token_type_embeddings.weight.detach().clone()
    te.embeddings = te.module.embeddings

    class _Cfg(dict):
        __getattr__ = dict.__getitem__
    te.original_config = _Cfg(num_segments=5)
    te.config = cfg
    torch.manual_seed(64)
    te._init_segment_embeddings()
    te.eval()
    B, T = 3, 12
    ids = torch.randint(0, 50, (B, T), generator=g)
    mask = torch.ones(B, T, dtype=torch.long)
    mask[1, 7:] = 0
    seg = torch.randint(0, 5, (B, T), generator=g)
    pooled = te(ids, mask, seg)
    seq = te(ids, mask, seg, return_sequence=True)
    w = torch.randn(seq.shape, generator=g)
    wp = torch.randn(pooled.shape, generator=g)
    ((seq * w).sum() + (pooled * wp).sum()).backward()
    names = [n for n, _ in te.named_parameters()]
    _save("encoders", {
        "fc7": {"state_dict": {k: v.detach().clone() for k, v in fc7.state_dict().items()}, "feat": feat.detach(),
                "out": y.detach(), "w_rand": wy, "dfeat": feat.grad.detach(),
                "grads": {"lc.weight": fc7.lc.weight.grad.clone(), "lc.bias": fc7.lc.bias.grad.clone()},
                "legacy_keys": sorted(legacy.keys())},
        "transformer": {"cfg": {"hidden": 128, "heads": 2, "inter": 256, "layers": 2, "vocab": 50, "max_pos": 32,
                                "num_segments": 5},
                        "pre_types": pre_types,
                        "state_dict": {k: v.detach().clone() for k, v in te.state_dict().items()},
                        "ids": ids, "mask": mask, "seg": seg, "seq": seq.detach(), "pooled": pooled.detach(),
                        "w_seq": w, "w_pooled": wp, "grads": _grads(te, names)},
    })


def golden_uniter():
    """UNITERModelBase.forward (uniter.py:197-243) with UNITERImageEmbeddings (:43-88).  The constructor pulls
    bert-base-uncased from the hub, so the object is assembled around the reference's own forward / embedding code with
    explicit-config sub-modules; the encoder is the reference's BertEncoderJit (what replace_with_jit() installs)."""
    from transformers import BertConfig
    from transformers.models.bert.modeling_bert import BertEmbeddings, BertPooler
    un = R.uniter()
    hl = R.hf_layers()
    cfg = BertConfig(hidden_size=128, num_attention_heads=2, intermediate_size=256, num_hidden_layers=2, vocab_size=50,
                     max_position_embeddings=32, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    m = un.UNITERModelBase.__new__(un.UNITERModelBase)
    torch.nn.Module.__init__(m)
    m.text_embeddings = BertEmbeddings(cfg)
    m.img_embeddings = un.UNITERImageEmbeddings(img_dim=40, hidden_size=128, hidden_dropout_prob=0.0)
    m.encoder = hl.BertEncoderJit(cfg)
    m.pooler = BertPooler(cfg)
    _perturb(m, 81)
    m.eval()
    g = torch.Generator().manual_seed(82)
    B, T, Rr = 3, 6, 5
    ids = torch.randint(0, 50, (B, T), generator=g)
    pos_ids = torch.arange(T).unsqueeze(0).expand(B, T).contiguous()
    feat = torch.randn(B, Rr, 40, generator=g, requires_grad=True)
    pos = torch.rand(B, Rr, 7, generator=g)
    att = torch.ones(B, T + Rr, dtype=torch.long)
    att[1, 4:T] = 0
    att[2, T + 3:] = 0
    img_masks = torch.zeros(B, Rr, dtype=torch.long)
    img_masks[0, 1] = 1
    out = m(ids, pos_ids, feat, pos, att)
    w = torch.randn(out.final_layer.shape, generator=g)
    (out.final_layer * w).sum().backward()
    names = [n for n, _ in m.named_parameters()]
    masked = m(ids, pos_ids, feat.detach(), pos, att, img_masks=img_masks).final_layer.detach()
    img_only = m(ids, pos_ids, feat.detach(), pos, att[:, T:], input_modality="image").final_layer.detach()
    _save("uniter", {
        "cfg": {"hidden": 128, "heads": 2, "inter": 256, "layers": 2, "vocab": 50, "max_pos": 32, "img_dim": 40},
        "state_dict": {k: v.detach().clone() for k, v in m.state_dict().items()},
        "ids": ids, "pos_ids": pos_ids, "feat": feat.detach(), "pos": pos, "att": att, "img_masks": img_masks,
        "final": out.final_layer.detach(), "n_hidden": len(out.hidden_layers),
        "hidden_1": out.hidden_layers[1].detach(), "w_rand": w, "dfeat": feat.grad.detach(), "grads": _grads(m, names),
        "final_masked": masked, "final_image_only": img_only,
    })


def golden_lxmert():
    """LXMERTEncoder.forward (lxmert.py:309-336) = VisualFeatEncoder + language / relational BERT layers + cross-modality
    layers with the shared cross-attention block, under the reference's replace_with_jit() (lxmert.py relies on
    BertSelfAttention(encoder_hidden_states=...), which only the reference's JIT forwards provide on transformers 5)."""
    from transformers import BertConfig
    hl = R.hf_layers()
    lx = R.lxmert()
    cfg = BertConfig(hidden_size=64, num_attention_heads=1, intermediate_size=128, vocab_size=50,
                     hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    cfg.visual_feat_dim, cfg.visual_pos_dim, cfg.l_layers, cfg.x_layers, cfg.r_layers = 40, 4, 2, 2, 1
    hl.replace_with_jit()
    try:
        enc = lx.LXMERTEncoder(cfg).eval()
        _perturb(enc, 91)
        g = torch.Generator().manual_seed(92)
        B, T, Rr = 3, 7, 5
        lang = torch.randn(B, T, 64, generator=g, requires_grad=True)
        feats = torch.randn(B, Rr, 40, generator=g, requires_grad=True)
        boxes = torch.rand(B, Rr, 4, generator=g)
        lmask = torch.ones(B, T, dtype=torch.long)
        lmask[1, 4:] = 0
        vmask = torch.ones(B, Rr, dtype=torch.long)
        vmask[2, 3:] = 0
        ladd = (1.0 - lmask[:, None, None, :].float()) * -10000.0
        vadd = (1.0 - vmask[:, None, None, :].float()) * -10000.0
        lo, vo = enc(lang, ladd, (feats, boxes), vadd)
        wl, wv = torch.randn(lo.shape, generator=g), torch.randn(vo.shape, generator=g)
        ((lo * wl).sum() + (vo * wv).sum()).backward()
        names = [n for n, _ in enc.named_parameters()]
        _save("lxmert", {
            "cfg": {"hidden": 64, "heads": 1, "inter": 128, "feat_dim": 40, "pos_dim": 4, "l": 2, "x": 2, "r": 1},
            "state_dict": {k: v.detach().clone() for k, v in enc.state_dict().items()},
            "lang": lang.detach(), "feats": feats.detach(), "boxes": boxes, "lmask": lmask, "vmask": vmask,
            "lang_out": lo.detach(), "visn_out": vo.detach(), "wl": wl, "wv": wv, "dlang": lang.grad.detach(),
            "dfeats": feats.grad.detach(), "grads": _grads(enc, names),
        })
    finally:
        hl.undo_replace_with_jit()


def golden_mlm_head():
    """`self.cls` of VisualBERTForPretraining (visual_bert.py:205-214) = HF BertPreTrainingHeads with the decoder tied to
    the word embeddings, and the masked-LM loss (:269-277).  Third-party arithmetic (transformers): the installed
    module is run as is; keys are stored with the reference pin's names (`predictions.bias` is the decoder bias)."""
    from transformers import BertConfig
    from transformers.models.bert.modeling_bert import BertPreTrainingHeads
    cfg = BertConfig(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=1, vocab_size=203)
    heads = BertPreTrainingHeads(cfg)
    emb = torch.nn.Embedding(203, 64)
    heads.predictions.decoder.weight = emb.weight
    _perturb(heads, 95)
    heads.eval()
    g = torch.Generator().manual_seed(96)
    B, S = 3, 9
    seq = torch.randn(B, S, 64, generator=g, requires_grad=True)
    pooled = torch.randn(B, 64, generator=g)
    labels = torch.full((B, S), -1, dtype=torch.long)
    labels[0, 2], labels[0, 5], labels[1, 1], labels[2, 7] = 17, 202, 0, 99
    scores, rel_score = heads(seq, pooled)
    loss = torch.nn.CrossEntropyLoss(ignore_index=-1)(scores.view(-1, 203), labels.view(-1))
    loss.backward()
    sd = {"cls.predictions.transform.dense.weight": heads.predictions.transform.dense.weight,
          "cls.predictions.transform.dense.bias": heads.predictions.transform.dense.bias,
          "cls.predictions.transform.LayerNorm.weight": heads.predictions.transform.LayerNorm.weight,
          "cls.predictions.transform.LayerNorm.bias": heads.predictions.transform.LayerNorm.bias,
          "cls.predictions.decoder.weight": heads.predictions.decoder.weight,
          "cls.predictions.bias": heads.predictions.decoder.bias,
          "cls.seq_relationship.weight": heads.seq_relationship.weight,
          "cls.seq_relationship.bias": heads.seq_relationship.bias}
    _save("mlm_head", {
        "cfg": {"hidden": 64, "vocab": 203}, "state_dict": {k: v.detach().clone() for k, v in sd.items()},
        "seq": seq.detach(), "pooled": pooled, "labels": labels, "scores": scores.detach(), "rel": rel_score.detach(),
        "loss": loss.detach(), "dseq": seq.grad.detach(),
        "grads": {k: v.grad.detach().clone() for k, v in sd.items() if v.grad is not None},
    })


def golden_visual_bert_bypass():
    """VisualBERTBase.forward with bypass_transformer=True (visual_bert.py:118-143): the encoder sees the text only, one
    `additional_layer` fuses [text output; visual embeddings].  Also the plain path of the same class for reference."""
    from transformers import BertConfig
    vb = R.visual_bert()
    orig = vb.VisualBERTBase.init_weights
    vb.VisualBERTBase.init_weights = lambda self: None            # see ref_loader.visual_bert()
    try:
        cfg = BertConfig(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=2, vocab_size=51,
                         max_position_embeddings=64, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
        m = vb.VisualBERTBase(cfg, visual_embedding_dim=40, bypass_transformer=True).eval()
    finally:
        vb.VisualBERTBase.init_weights = orig
    _perturb(m, 97)
    g = torch.Generator().manual_seed(98)
    B, T, Rr = 3, 8, 4
    ids = torch.randint(1, 51, (B, T), generator=g)
    seg = torch.zeros(B, T, dtype=torch.long)
    feats = torch.randn(B, Rr, 40, generator=g, requires_grad=True)
    vtype = torch.zeros(B, Rr, dtype=torch.long)
    att = torch.ones(B, T + Rr, dtype=torch.long)
    att[1, 5:T] = 0
    att[2, T + 2:] = 0
    seq, pooled, _ = m(ids, att, seg, feats, vtype)
    w = torch.randn(seq.shape, generator=g)
    (seq * w).sum().backward()
    names = [n for n, _ in m.named_parameters()]
    m.bypass_transformer = False
    plain_seq, plain_pooled, _ = m(ids, att, seg, feats.detach(), vtype)
    _save("visual_bert_bypass", {
        "cfg": {"hidden": 64, "heads": 1, "inter": 128, "layers": 2, "vocab": 51, "max_pos": 64, "vdim": 40},
        "state_dict": {k: v.detach().clone() for k, v in m.state_dict().items()},
        "ids": ids, "seg": seg, "feats": feats.detach(), "vtype": vtype, "att": att, "seq": seq.detach(),
        "pooled": pooled.detach(), "w_rand": w, "dfeats": feats.grad.detach(), "grads": _grads(m, names),
        "plain_seq": plain_seq.detach(), "plain_pooled": plain_pooled.detach(),
    })


def golden_adamw():
    """optimizer `adam_w`: 5 steps on three small parameters, two hyper-parameter groups (decay / no decay), with the
    reference's transformers arithmetic (AdamWSkipParamsWithZeroGrad.step, optimizers.py:22-86) and with what `adam_w`
    itself resolves to here (torch.optim.AdamW, optimizers.py:8-14)."""
    opt = R.optimizers()
    g = torch.Generator().manual_seed(71)
    init = [torch.randn(16, 24, generator=g), torch.randn(24, generator=g), 1.0 + 0.1 * torch.randn(24, generator=g)]
    grads = [[torch.randn(t.shape, generator=g) * 0.1 for t in init] for _ in range(5)]
    hp = dict(lr=5e-3, betas=(0.9, 0.98), eps=1e-6)

    def run(cls):
        ps = [torch.nn.Parameter(t.clone()) for t in init]
        o = cls([{"params": [ps[0]], "weight_decay": 0.01}, {"params": ps[1:], "weight_decay": 0.0}], **hp)
        traj = []
        for gs in grads:
            for p_, g_ in zip(ps, gs):
                p_.grad = g_.clone()
            o.step()
            traj.append([p_.detach().clone() for p_ in ps])
        return traj
    _save("adamw", {"init": init, "grads": grads, "hp": hp, "weight_decay": [0.01, 0.0, 0.0],
                    "transformers": run(opt.AdamWSkipParamsWithZeroGrad), "torch": run(opt.AdamW),
                    "adam_w_is": opt.AdamW.__module__})


def golden_vit():
    """ViTEncoder (pre-LN blocks with a key-padding mask, mmf/modules/vit.py:63-175) and the ViTModel tail (final LayerNorm +
    pooler, vit.py:178-274) fed already-embedded tokens (`do_patch_embeddings=False`, the ViLT use, vit.py:187) and pixel
    values (HF ViTEmbeddings: patch conv + [CLS] + position table)."""
    from transformers import ViTConfig
    import transformers.models.vit.modeling_vit as hv
    vit = R.vit()
    cfg = ViTConfig(hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=256,
                    hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, image_size=32, patch_size=8,
                    layer_norm_eps=1e-12)           # head size 64: the attention kernels take 64 or 128
    cfg.chunk_size_feed_forward, cfg.is_decoder, cfg.position_embedding_type, cfg.max_position_embeddings = 0, False, "absolute", 64
    enc = vit.ViTEncoder(cfg).eval()
    _perturb(enc, 91)
    with torch.no_grad():                               # _perturb's LayerNorm rule keys on "LayerNorm.weight": ViT's are
        for n, p_ in enc.named_parameters():            # `layernorm_before/after.weight`
            if "layernorm" in n and n.endswith("weight"):
                p_.add_(1.0)
    g = torch.Generator().manual_seed(92)
    B, S = 3, 17
    x = torch.randn(B, S, 128, generator=g, requires_grad=True)
    mask = torch.ones(B, S, dtype=torch.long)
    mask[1, 12:] = 0
    add = (1.0 - mask[:, None, None, :].float()) * -10000.0
    out = enc(x, attention_mask=add, output_hidden_states=True, return_dict=False)
    w = torch.randn(out[0].shape, generator=g)
    (out[0] * w).sum().backward()
    names = [n for n, _ in enc.named_parameters()]
    # model tail + embeddings from pixels
    emb = hv.ViTEmbeddings(cfg).eval()
    ln = torch.nn.LayerNorm(128, eps=1e-12)
    pool = hv.ViTPooler(cfg).eval()
    for m_, sd_ in ((emb, 93), (ln, 94), (pool, 95)):
        _perturb(m_, sd_)
    with torch.no_grad():
        ln.weight.add_(1.0)
        emb.cls_token.copy_(torch.randn(emb.cls_token.shape, generator=g) * 0.02)
        emb.position_embeddings.copy_(torch.randn(emb.position_embeddings.shape, generator=g) * 0.02)
    pix = torch.randn(B, 3, 32, 32, generator=g)
    with torch.no_grad():
        e = emb(pix)
        seq = ln(enc(e, attention_mask=None, return_dict=False)[0])
        pooled = pool(seq)
    sd = {"encoder." + k: v.detach().clone() for k, v in enc.state_dict().items()}
    sd.update({"embeddings." + k: v.detach().clone() for k, v in emb.state_dict().items()})
    sd.update({"layernorm." + k: v.detach().clone() for k, v in ln.state_dict().items()})
    sd.update({"pooler." + k: v.detach().clone() for k, v in pool.state_dict().items()})
    _save("vit", {
        "cfg": {"hidden": 128, "heads": 2, "inter": 256, "layers": 2, "image_size": 32, "patch_size": 8},
        "state_dict": sd, "x": x.detach(), "mask": mask, "out": out[0].detach(), "hidden_1": out[1][1].detach(),
        "n_hidden": len(out[1]), "w_rand": w, "dx": x.grad.detach(),
        "grads": {"encoder." + k: v for k, v in _grads(enc, names).items()},
        "pixels": pix, "embedded": e, "seq_from_pixels": seq, "pooled_from_pixels": pooled,
    })


def golden_vinvl():
    """VinVLBase.forward (vinvl.py:43-122), with the 2054-wide VinVL region features scaled down to 46 (46 % 8 = 6, like
    2054 % 8 = 6: the column padding of the GEMM is exercised the same way)."""
    from transformers import BertConfig
    vv = R.vinvl()
    cfg = BertConfig(hidden_size=128, num_attention_heads=2, intermediate_size=256, num_hidden_layers=2, vocab_size=50,
                     max_position_embeddings=32, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    cfg.img_feature_dim, cfg.use_img_layernorm, cfg.img_layer_norm_eps = 46, True, 1e-12
    m = vv.VinVLBase(cfg).eval()
    # with the pinned transformers (<= 4.10) HF's BertEncoder honours output_hidden_states; transformers 5 moved that into
    # model-level hooks, so the encoder runs under the reference's own replace_with_jit() (BertEncoderJit.forward,
    # hf_layers.py:316-355 - the implementation MMF installs process-wide from its model constructors)
    hl = R.hf_layers()
    hl.replace_with_jit()
    try:
        return _golden_vinvl_body(m)
    finally:
        hl.undo_replace_with_jit()


def _golden_vinvl_body(m):
    _perturb(m, 171)
    with torch.no_grad():
        m.img_embedding[1].weight.add_(1.0)           # "img_embedding.1.weight" is a LayerNorm scale
    g = torch.Generator().manual_seed(172)
    B, T, Rr = 3, 7, 5
    ids = torch.randint(1, 50, (B, T), generator=g)
    feats = torch.randn(B, Rr, 46, generator=g, requires_grad=True)
    att = torch.ones(B, T + Rr, dtype=torch.long)
    att[1, 5:T] = 0
    att[2, T + 3:] = 0
    out = m(ids, feats, attention_mask=att)
    w = torch.randn(out.last_hidden_state.shape, generator=g)
    (out.last_hidden_state * w).sum().backward()
    names = [n for n, p_ in m.named_parameters() if p_.grad is not None]
    _save("vinvl", {
        "cfg": {"hidden": 128, "heads": 2, "inter": 256, "layers": 2, "vocab": 50, "max_pos": 32, "img_dim": 46},
        "state_dict": {k: v.detach().clone() for k, v in m.state_dict().items() if v.dtype.is_floating_point},
        "ids": ids, "feats": feats.detach(), "att": att, "last": out.last_hidden_state.detach(),
        "n_hidden": len(out.hidden_layers), "hidden_1": out.hidden_layers[1].detach(), "w_rand": w,
        "dfeats": feats.grad.detach(), "grads": _grads(m, names)})


class _OmegaConfShim:
    """the two OmegaConf calls the reference's model classes make on this path (visual_bert.py:171-173, vilbert.py:1061-1063)"""

    @staticmethod
    def to_container(cfg, resolve=True):
        return dict(cfg)


def _new_base_model(cls, cfg):
    """BaseModel is lightning-backed in the reference (not importable here): build the registered model class around a
    plain nn.Module base - its build() / forward() are the reference's own."""
    m = cls.__new__(cls)
    torch.nn.Module.__init__(m)
    m.config = cfg
    return m


def _ref_model_modules():
    R._install()
    R.load("mmf/utils/transform.py", "mmf.utils.transform")
    R.load("mmf/utils/torchscript.py", "mmf.utils.torchscript")
    vb, vil = R.visual_bert(), R.vilbert()
    for mod in (vb, vil):
        mod.OmegaConf = _OmegaConfShim
        mod.get_mmf_cache_dir = lambda: "/tmp"
    vb.VisualBERTBase.init_weights = lambda self: None          # see ref_loader.visual_bert()
    vil.ViLBERTBase.init_weights = lambda self: None
    vil.ViLBERTBase.from_pretrained = classmethod(lambda cls, name, config=None, cache_dir=None, **kw: cls(config, **kw))
    return vb, vil


def golden_models():
    """The reference's REGISTERED MODEL classes end to end: VisualBERT / ViLBERT `forward(sample_list)` -> scores / losses
    (visual_bert.py:407-601, vilbert.py:1336-1472), classification and pretraining heads, plus the integer tensors the
    SampleList plumbing derives (image_mask, attention_mask, padded labels)."""
    vb, vil = _ref_model_modules()
    g = torch.Generator().manual_seed(123)
    out = {}
    # ---------------- VisualBERT ----------------
    base = dict(bert_model_name=None, visual_embedding_dim=40, special_visual_initialize=True, embedding_strategy="plain",
                bypass_transformer=False, output_attentions=False, output_hidden_states=False, random_initialize=True,
                freeze_base=False, finetune_lr_multiplier=1, pooler_strategy="default", zerobias=False, num_labels=3,
                hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=2, vocab_size=51,
                max_position_embeddings=64, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    B, T, Rr = 4, 8, 5
    ids = torch.randint(1, 51, (B, T), generator=g)
    mask = torch.ones(B, T, dtype=torch.long)
    mask[1, 6:] = 0
    mask[3, 4:] = 0
    seg = torch.zeros(B, T, dtype=torch.long)
    feats = torch.randn(B, Rr, 40, generator=g).abs()
    maxf = torch.tensor([5, 2, 3, 4])
    labels = torch.full((B, T), -1)
    labels[0, 2], labels[1, 4], labels[2, 1], labels[2, 6] = 7, 11, 3, 40
    targets = torch.tensor([0, 2, 1, 1])

    def sample_list():
        return _Cfg(input_ids=ids.clone(), input_mask=mask.clone(), segment_ids=seg.clone(), image_feature_0=feats.clone(),
                    image_info_0=_Cfg(max_features=maxf.clone()), lm_label_ids=labels.clone(), targets=targets.clone(),
                    dataset_name="golden", dataset_type="train")

    for head, strategy in (("classification", "default"), ("classification", "vqa"), ("pretraining", "default")):
        cfg = _Cfg(dict(base, training_head_type=head, pooler_strategy=strategy))
        m = _new_base_model(vb.VisualBERT, cfg)
        m.training_head_type = head
        m.build()
        m.eval()
        _perturb(m, 500 + len(out))
        if head == "pretraining":
            # tie_weights() (visual_bert.py:227-235): transformers 5 no longer has _tie_or_clone_weights; its non-torchscript
            # branch is exactly this parameter sharing
            m.model.cls.predictions.decoder.weight = m.model.bert.embeddings.word_embeddings.weight
        sl = sample_list()
        o = m.forward(sl)
        if head == "classification":
            loss = torch.nn.functional.cross_entropy(o["scores"], targets)
        else:
            loss = o["losses"]["golden/train/masked_lm_loss"]
        loss.backward()
        names = [n for n, p_ in m.named_parameters() if p_.grad is not None]
        key = "visual_bert_%s_%s" % (head, strategy)
        out[key] = {
            "config": dict(cfg), "state_dict": {k: v.detach().clone() for k, v in m.state_dict().items()},
            "image_mask": sl["image_mask"], "attention_mask": sl["attention_mask"],
            "masked_lm_labels": sl["masked_lm_labels"] if head == "pretraining" else None,
            "scores": o["scores"].detach() if "scores" in o else None,
            "logits": o["logits"].detach() if "logits" in o else None, "loss": loss.detach(),
            "loss_keys": sorted(o.get("losses", {}).keys()), "grads": _grads(m, names)}
    out["visual_bert_inputs"] = {"ids": ids, "mask": mask, "seg": seg, "feats": feats, "max_features": maxf,
                                 "lm_label_ids": labels, "targets": targets}
    # ---------------- ViLBERT ----------------
    vcfg = dict(bert_model_name=None, num_labels=3, random_initialize=True, hidden_size=64, num_attention_heads=1,
                intermediate_size=128, num_hidden_layers=2, vocab_size=51, max_position_embeddings=64, type_vocab_size=2,
                hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, hidden_act="gelu", v_feature_size=40,
                v_target_size=17, v_hidden_size=64, v_num_hidden_layers=2, v_num_attention_heads=1, v_intermediate_size=96,
                bi_hidden_size=64, bi_num_attention_heads=1, bi_intermediate_size=64, bi_attention_type=1,
                v_attention_probs_dropout_prob=0.0, v_hidden_act="gelu", v_hidden_dropout_prob=0.0, v_initializer_range=0.02,
                v_biattention_id=[0, 1], t_biattention_id=[0, 1], pooling_method="mul", fusion_method="mul", fast_mode=False,
                with_coattention=True, dynamic_attention=False, in_batch_pairs=False, task_specific_tokens=False,
                fixed_v_layer=0, fixed_t_layer=0, visualization=False, visual_target=0, objective=0, num_negative=128,
                model="bert", layer_norm_eps=1e-12, initializer_range=0.02, output_attentions=False,
                output_hidden_states=False, freeze_base=False)
    bbox = torch.rand(B, Rr, 5, generator=g)
    cls_prob = torch.softmax(torch.randn(B, Rr, 17, generator=g), dim=-1)
    image_labels = torch.tensor([[1, 0, 0, 1, 0], [0, 1, 0, 0, 0], [0, 0, 0, 0, 1], [1, 1, 0, 0, 0]])
    for head in ("classification", "pretraining"):
        cfg = _Cfg(dict(vcfg, training_head_type=head))
        m = _new_base_model(vil.ViLBERT, cfg)
        m.build()
        m.eval()
        _perturb(m, 600 + len(out))
        sl = sample_list()
        sl["image_info_0"] = _Cfg(max_features=maxf.clone(), bbox=bbox.clone(), cls_prob=cls_prob.numpy().copy())
        sl["image_labels"] = image_labels.clone()
        o = m.forward(sl)
        if head == "classification":
            loss = torch.nn.functional.cross_entropy(o["scores"], targets)
        else:
            loss = sum(v.sum() for v in o["losses"].values())
        loss.backward()
        names = [n for n, p_ in m.named_parameters() if p_.grad is not None]
        out["vilbert_" + head] = {
            "config": dict(cfg), "state_dict": {k: v.detach().clone() for k, v in m.state_dict().items()},
            "scores": o["scores"].detach() if "scores" in o else None,
            "losses": {k: v.detach() for k, v in o.get("losses", {}).items()}, "loss": loss.detach(),
            "grads": _grads(m, names), "unused": sorted(n for n, p_ in m.named_parameters() if p_.grad is None)}
    out["vilbert_inputs"] = {"bbox": bbox, "cls_prob": cls_prob, "image_labels": image_labels}
    _save("models", out)


# the reference YAML files that MODEL_DEFAULTS (mmf_b200/models.py) restates, and those the config-loading test reads
MODEL_CONFIG_FILES = ["configs/models/visual_bert/defaults.yaml", "configs/models/vilbert/defaults.yaml",
                      "configs/models/mmbt/defaults.yaml", "configs/models/mmf_transformer/defaults.yaml",
                      "configs/models/visual_bert/classification.yaml", "configs/models/mmbt/classification.yaml",
                      "configs/models/mmbt/with_features.yaml"]


def golden_model_configs():
    """The parsed documents (yaml.safe_load, nothing resolved) of MODEL_CONFIG_FILES, keyed by their path under mmf/."""
    import yaml
    docs = {}
    for rel in MODEL_CONFIG_FILES:
        with open(os.path.join(R.REF_ROOT, "mmf", rel)) as fh:
            docs[rel] = yaml.safe_load(fh)
    path = os.path.join(OUT, "model_configs.json")
    with open(path, "w") as fh:
        json.dump(docs, fh, indent=1)
        fh.write("\n")
    print("wrote %s" % path)


def main():
    torch.manual_seed(0)
    torch.set_num_threads(4)
    golden_bert_encoder()
    golden_vilbert_encoder()
    golden_embeddings()
    golden_mmbt()
    golden_mmft_embeddings()
    golden_encoders()
    golden_adamw()
    golden_uniter()
    golden_lxmert()
    golden_mlm_head()
    golden_visual_bert_bypass()
    golden_models()
    golden_vit()
    golden_vinvl()
    golden_model_configs()


if __name__ == "__main__":
    main()
