"""Host orchestration of the fusion block on the CPU: mmf_b200.engine run over tests/fake_kernels.py (a torch restatement
of every kernel's CONTRACT) must reproduce the oracle - forward, input gradient and every parameter gradient in the flat
buffer - for a BERT layer stack and a ViLBERT connection layer, with and without dropout (same explicit masks on both
sides).  This pins which operand goes to which kernel, what is saved, and where gradients accumulate; the kernels
themselves are checked on the B200 (`-m gpu`)."""
import types

import pytest
import torch

from mmf_b200 import engine as E
from oracle import fusion_oracle as O
from oracle import golden_io

import fake_kernels as FK


@pytest.fixture()
def fake(monkeypatch):
    monkeypatch.setattr(E, "F", FK)
    yield FK


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-3 * b.numel() ** 0.5)).item()


def _bf16_round_(module):
    with torch.no_grad():
        for p in module.parameters():
            p.copy_(p.to(torch.bfloat16).float())


def _cfg(p):
    return types.SimpleNamespace(hidden_size=64, num_attention_heads=2, intermediate_size=128, num_hidden_layers=2,
                                 hidden_dropout_prob=p, attention_probs_dropout_prob=p, layer_norm_eps=1e-12)


class _RecordingDropout(E.DropoutState):
    """hands out the keep bits and remembers them in draw order, so that the oracle can be given the same masks"""

    def __init__(self):
        super().__init__(7)
        self.drawn = []

    def bits(self, rows_shape, ncols, p, device):
        w = super().bits(rows_shape, ncols, p, device)
        self.drawn.append((w, ncols))
        return w


@pytest.mark.parametrize("p", [0.0, 0.25])
def test_bert_layer_stack_wiring_matches_oracle(fake, p):
    from mmf_b200.modules import B200BertEncoder
    torch.manual_seed(0)
    enc = B200BertEncoder(_cfg(p))
    with torch.no_grad():
        for prm in enc.parameters():
            if prm.dim() == 1:
                prm.add_(torch.randn_like(prm) * 0.05)
    _bf16_round_(enc)
    params = []
    for m in enc.layer:
        params += E.BertLayerW.params(m)
    pack = E.ParamPack(params, "cpu")
    pack.refresh()
    weights = [E.BertLayerW(pack, m) for m in enc.layer]
    B, S, H = 3, 10, 64
    x = torch.randn(B, S, H).to(torch.bfloat16)
    mask = torch.ones(B, S, dtype=torch.long)
    mask[1, 6:] = 0
    add2d = ((1.0 - mask.float()) * -10000.0).contiguous()
    ds = _RecordingDropout() if p > 0 else None
    h = x.reshape(B * S, H)
    saved = []
    for w in weights:
        h, s = E.bert_layer_fwd(h, add2d, w, B, S, p, p, ds)
        saved.append(s)
    w_rand = torch.randn(B * S, H)
    pack.prepare_grads()
    d = w_rand.to(torch.bfloat16)
    for w, s in zip(reversed(weights), reversed(saved)):
        d = E.bert_layer_bwd(d, s, add2d, w, B, S)
    # ---- oracle on the same (bf16-rounded) weights, inputs and masks ----
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in enc.state_dict().items()}
    xo = x.float().clone().requires_grad_(True)
    masks = None
    if p > 0:
        it = iter(ds.drawn)
        masks = []
        for _ in weights:      # draw order of bert_layer_fwd: attention probs, attention output, FFN output
            a, n = next(it)
            so, n1 = next(it)
            fo, n2 = next(it)
            masks.append({"attn": FK.unpack_keep_bits(a, n), "self_out": FK.unpack_keep_bits(so, n1).view(B, S, n1),
                          "out": FK.unpack_keep_bits(fo, n2).view(B, S, n2)})
    out = O.bert_encoder(xo, O.extended_attention_mask(mask), sd, "", 2, 2, masks, p, p)
    (out.reshape(B * S, H) * w_rand.to(torch.bfloat16).float()).sum().backward()
    assert rel(h.float(), out.reshape(B * S, H)) < 2e-2
    assert rel(d.float(), xo.grad.reshape(B * S, H)) < 3e-2
    named = dict(enc.named_parameters())
    for k, v in sd.items():
        if ".key.bias" in k:
            continue            # analytically zero
        assert rel(pack.grad_view(named[k]), v.grad) < 3e-2, k


def test_vilbert_connection_layer_wiring_matches_oracle(fake):
    from mmf_b200.modules import B200ViLBertEncoder
    torch.manual_seed(1)
    c = dict(hidden_size=64, num_attention_heads=2, intermediate_size=128, num_hidden_layers=1,
             v_hidden_size=128, v_num_attention_heads=2, v_intermediate_size=128, v_num_hidden_layers=1,
             bi_hidden_size=128, bi_num_attention_heads=2, v_biattention_id=[0], t_biattention_id=[0])
    cfg = types.SimpleNamespace(hidden_dropout_prob=0.0, v_hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                                v_attention_probs_dropout_prob=0.0, layer_norm_eps=1e-12, **c)
    enc = B200ViLBertEncoder(cfg)
    _bf16_round_(enc)
    m = enc.c_layer[0]
    used = E.ConnectionW.params(m)
    pack = E.ParamPack(used, "cpu")
    pack.refresh()
    w = E.ConnectionW(pack, m)
    B, R, T = 2, 5, 7
    img = torch.randn(B * R, 128).to(torch.bfloat16)
    txt = torch.randn(B * T, 64).to(torch.bfloat16)
    imask = torch.ones(B, R, dtype=torch.long)
    tmask = torch.ones(B, T, dtype=torch.long)
    tmask[0, 4:] = 0
    iadd = ((1.0 - imask.float()) * -10000.0).contiguous()
    tadd = ((1.0 - tmask.float()) * -10000.0).contiguous()
    o1, o2, saved = E.connection_fwd(img, txt, iadd, tadd, w, B, R, T, 0.0, 0.0, 0.0, 0.0, None)
    wv, wt = torch.randn(B * R, 128), torch.randn(B * T, 64)
    pack.prepare_grads()
    dimg, dtxt = E.connection_bwd(wv.to(torch.bfloat16), wt.to(torch.bfloat16), saved, iadd, tadd, w, B, R, T)
    sd = {"c." + k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    io = img.float().view(B, R, 128).clone().requires_grad_(True)
    to = txt.float().view(B, T, 64).clone().requires_grad_(True)
    ov, ot = O.connection_layer(io, O.extended_attention_mask(imask), to, O.extended_attention_mask(tmask), sd, "c", 2)
    ((ov.reshape(B * R, 128) * wv.to(torch.bfloat16).float()).sum() + (ot.reshape(B * T, 64) * wt.to(torch.bfloat16).float()).sum()).backward()
    assert rel(o1.float(), ov.reshape(B * R, 128)) < 2e-2 and rel(o2.float(), ot.reshape(B * T, 64)) < 2e-2
    assert rel(dimg.float(), io.grad.reshape(B * R, 128)) < 3e-2 and rel(dtxt.float(), to.grad.reshape(B * T, 64)) < 3e-2
    named = dict(m.named_parameters())
    for k, prm in named.items():
        g = sd["c." + k].grad
        if g is None:
            continue            # biOutput.q_dense1/2: unused in the reference too
        if "key" in k and k.endswith("bias"):
            continue
        assert rel(pack.grad_view(prm), g) < 3e-2, k


# ---------------------------------------------------------------------------------------------------------------
# the drop-in modules end to end (autograd Function, parameter pack hand-over, ViLBERT schedule) over the test double,
# against the reference's own outputs (tests/golden)
# ---------------------------------------------------------------------------------------------------------------


@pytest.fixture()
def cpu_modules(fake, monkeypatch):
    import mmf_b200.modules as M
    monkeypatch.setattr(M, "_require_cuda", lambda t, what: None)
    yield M


def _golden_bound(e, tol=4e-2):
    # bf16 weights / activations against the reference's fp32 run on a 10-token fixture (see test_encoder_gpu.py)
    return e < tol


def test_bert_encoder_module_vs_reference_golden_cpu(cpu_modules):
    g = golden_io.load("bert_encoder")
    c = g["cfg"]
    cfg = types.SimpleNamespace(hidden_size=c["hidden"], num_attention_heads=c["heads"], intermediate_size=c["inter"],
                                num_hidden_layers=c["layers"], hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                                layer_norm_eps=1e-12)
    enc = cpu_modules.B200BertEncoder(cfg)
    enc.load_state_dict(g["state_dict"])
    enc.eval()
    x = g["x"].clone().requires_grad_(True)
    add = O.extended_attention_mask(g["mask"])
    out = enc(x, add)[0]
    assert out.dtype == x.dtype and torch.isfinite(out).all()
    assert _golden_bound(rel(out, g["out"]), 2e-2)
    (out * g["w_rand"]).sum().backward()
    assert _golden_bound(rel(x.grad, g["dx"]))
    named = dict(enc.named_parameters())
    for k, gv in g["grads"].items():
        if ".key.bias" in k:
            continue
        assert _golden_bound(rel(named[k].grad, gv)), k
    # gradients live in (and alias) the flat buffer
    p0 = named["layer.0.attention.self.query.weight"]
    assert p0.grad.data_ptr() == enc._runner.pack.grad_view(p0).data_ptr()


def test_bert_encoder_applied_twice_in_one_graph_cpu(cpu_modules):
    cfg = types.SimpleNamespace(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=1,
                                hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, layer_norm_eps=1e-12)
    torch.manual_seed(3)
    enc = cpu_modules.B200BertEncoder(cfg).eval()
    x1, x2 = torch.randn(2, 6, 64), torch.randn(2, 6, 64)
    w1, w2 = torch.randn(2, 6, 64), torch.randn(2, 6, 64)

    def grads(fn):
        enc.zero_grad(set_to_none=True)
        fn().backward()
        return {k: p.grad.detach().clone() for k, p in enc.named_parameters()}
    both = grads(lambda: (enc(x1, None)[0] * w1).sum() + (enc(x2, None)[0] * w2).sum())
    a = grads(lambda: (enc(x1, None)[0] * w1).sum())
    b = grads(lambda: (enc(x2, None)[0] * w2).sum())
    for k in both:
        assert rel(both[k], a[k] + b[k]) < 2e-2, k


def test_vilbert_encoder_module_vs_reference_golden_cpu(cpu_modules):
    g = golden_io.load("vilbert_encoder")
    cfg = types.SimpleNamespace(hidden_dropout_prob=0.0, v_hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                                v_attention_probs_dropout_prob=0.0, **dict(g["cfg"]))
    enc = cpu_modules.B200ViLBertEncoder(cfg)
    enc.load_state_dict(g["state_dict"])
    enc.eval()
    txt = g["txt"].clone().requires_grad_(True)
    img = g["img"].clone().requires_grad_(True)
    tadd, iadd = O.extended_attention_mask(g["tmask"]), O.extended_attention_mask(g["imask"])
    tl, vl, _ = enc(txt, img, tadd, tadd, iadd, None, output_all_encoded_layers=False)
    assert _golden_bound(rel(tl[-1], g["t_out"]), 2e-2) and _golden_bound(rel(vl[-1], g["v_out"]), 2e-2)
    ((tl[-1] * g["wt"]).sum() + (vl[-1] * g["wv"]).sum()).backward()
    assert _golden_bound(rel(txt.grad, g["dtxt"])) and _golden_bound(rel(img.grad, g["dimg"]))
    for n, p in enc.named_parameters():
        if n in g["unused"]:
            assert p.grad is None, n
        elif "key" in n and n.endswith("bias"):
            continue
        else:
            assert _golden_bound(rel(p.grad, g["grads"][n]), 8e-2), n
    # output_all_encoded_layers=True: one entry per co-attention block = the states right after that block, and NOT the
    # final states (vilbert.py:761-763, 787-790) - against the oracle's walk of the same schedule
    with torch.no_grad():
        tl_all, vl_all, _ = enc(g["txt"], g["img"], tadd, tadd, iadd, None, output_all_encoded_layers=True)
        c = dict(g["cfg"])
        assert len(tl_all) == len(vl_all) == len(c["v_biattention_id"])
        sd = {k: v.to(torch.bfloat16).float() for k, v in g["state_dict"].items()}
        t, v, k = g["txt"].to(torch.bfloat16).float(), g["img"].to(torch.bfloat16).float(), 0
        for kind, i in O.vilbert_schedule(c["v_biattention_id"], c["t_biattention_id"], c["num_hidden_layers"],
                                          c["v_num_hidden_layers"]):
            if kind == "t":
                t, _ = O.bert_layer(t, tadd, sd, "layer.%d" % i, c["num_attention_heads"])
            elif kind == "v":
                v, _ = O.bert_layer(v, iadd, sd, "v_layer.%d" % i, c["v_num_attention_heads"])
            else:
                v, t = O.connection_layer(v, iadd, t, tadd, sd, "c_layer.%d" % i, c["bi_num_attention_heads"])
                assert rel(tl_all[k], t) < 2e-2 and rel(vl_all[k], v) < 2e-2, k
                k += 1
        assert rel(tl_all[-1], g["t_out"]) > 1e-2        # the last entry is NOT the final state (trailing layers follow)


def test_train_mode_dropout_is_repeatable_under_manual_seed_cpu(cpu_modules):
    cfg = types.SimpleNamespace(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=2,
                                hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, layer_norm_eps=1e-12)
    torch.manual_seed(5)
    enc = cpu_modules.B200BertEncoder(cfg).train()
    x = torch.randn(2, 8, 64)

    def run():
        torch.manual_seed(11)
        cpu_modules._SEED_COUNTER[0] = 0
        return enc(x, None)[0].detach().clone()
    a, b = run(), run()
    assert torch.equal(a, b)
    enc.eval()
    assert not torch.equal(enc(x, None)[0], a)      # dropout was really applied in train mode


# ---------------------------------------------------------------------------------------------------------------
# front-ends (embedding composers, MMBT token surgery, MMFT backend embeddings, encoder plugins) over the test double
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture()
def cpu_frontends(cpu_modules, monkeypatch):
    import mmf_b200.embeddings as EM
    import mmf_b200.encoders as EN
    import mmf_b200.mmbt as MB
    import mmf_b200.mmft_backend as MF
    import mmf_b200.ops as OPS
    import mmf_b200.vilbert as VB
    monkeypatch.setattr(OPS, "F", FK)
    monkeypatch.setattr(EM, "F", FK)
    for mod in (EM, EN, MB, MF, VB):
        if hasattr(mod, "_require_cuda"):
            monkeypatch.setattr(mod, "_require_cuda", lambda t, what: None)
    yield types.SimpleNamespace(EM=EM, EN=EN, MB=MB, MF=MF, VB=VB)


def test_visio_linguistic_embeddings_vs_reference_golden_cpu(cpu_frontends):
    g = golden_io.load("embeddings")
    sd = g["vl_state_dict"]
    cfg = types.SimpleNamespace(hidden_size=sd["word_embeddings.weight"].shape[1],
                                vocab_size=sd["word_embeddings.weight"].shape[0],
                                max_position_embeddings=sd["position_embeddings.weight"].shape[0],
                                type_vocab_size=sd["token_type_embeddings.weight"].shape[0], hidden_dropout_prob=0.0,
                                visual_embedding_dim=sd["projection.weight"].shape[1], layer_norm_eps=1e-12)
    emb = cpu_frontends.EM.B200VisioLinguisticEmbeddings(cfg)
    emb.load_state_dict({k: v for k, v in sd.items() if k in emb.state_dict()}, strict=False)
    emb.eval()
    out = emb(g["ids"], g["seg"], g["feats"], g["vtype"])
    assert rel(out, g["out_plain"]) < 2e-2
    out = emb(g["ids"], g["seg"], g["feats"], g["vtype"], g["alignment"])
    assert rel(out, g["out_alignment"]) < 2e-2
    out = emb(g["ids"], g["seg"])
    assert rel(out, g["out_text"]) < 2e-2
    # [PAD] row of the word table: read in the forward, no gradient (nn.Embedding(padding_idx=0))
    ids = g["ids"].clone()
    ids[:, -2:] = 0
    emb.zero_grad(set_to_none=True)
    emb(ids, g["seg"], g["feats"], g["vtype"]).float().square().sum().backward()
    gw = emb.word_embeddings.weight.grad
    assert torch.count_nonzero(gw[0]) == 0 and torch.count_nonzero(gw) > 0


def test_mmbt_vs_reference_golden_cpu(cpu_frontends):
    g = golden_io.load("mmbt")
    c = g["cfg"]
    cfg = types.SimpleNamespace(hidden_size=c["hidden"], num_attention_heads=c["heads"], intermediate_size=c["inter"],
                                num_hidden_layers=c["layers"], hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1,
                                layer_norm_eps=1e-12, hidden_act="gelu", initializer_range=0.02, vocab_size=50,
                                max_position_embeddings=64, type_vocab_size=2, modal_hidden_size=c["modal_hidden"])
    base = cpu_frontends.MB.B200MMBTBase(cfg)
    base.mmbt.load_state_dict(g["state_dict"], strict=False)
    base.eval()
    sl = {"input_ids": g["ids"].clone(), "input_mask": g["mask"].clone(), "segment_ids": g["seg"],
          "image_feature_0": g["feats"]}
    seq, pooled, _ = base(sl)
    assert torch.equal(sl["input_ids"], g["shifted_ids"]) and torch.equal(sl["input_mask"], g["shifted_mask"])
    assert rel(seq, g["seq_out"]) < 2e-2 and rel(pooled, g["pooled"]) < 2e-2


def test_encoder_plugins_vs_reference_golden_cpu(cpu_frontends):
    g = golden_io.load("encoders")
    f = g["fc7"]
    fc7 = cpu_frontends.EN.B200FinetuneFasterRcnnFpnFc7({"in_dim": 256, "out_dim": 128})
    fc7.load_state_dict(f["state_dict"])
    x = f["feat"].clone().requires_grad_(True)
    y = fc7(x)
    assert rel(y, f["out"]) < 1e-2
    (y * f["w_rand"]).sum().backward()
    assert rel(x.grad, f["dfeat"]) < 6e-2 and rel(fc7.lc.weight.grad, f["grads"]["lc.weight"]) < 6e-2
    t = g["transformer"]
    c = t["cfg"]
    te = cpu_frontends.EN.B200TransformerEncoder(dict(
        hidden_size=c["hidden"], num_hidden_layers=c["layers"], num_attention_heads=c["heads"],
        intermediate_size=c["inter"], vocab_size=c["vocab"], max_position_embeddings=c["max_pos"],
        num_segments=c["num_segments"]))
    te.load_state_dict(t["state_dict"])
    te.eval()
    pooled = te(t["ids"], t["mask"], t["seg"])
    seq = te(t["ids"], t["mask"], t["seg"], return_sequence=True)
    assert rel(seq, t["seq"]) < 2e-2 and rel(pooled, t["pooled"]) < 2e-2
    ((seq * t["w_seq"]).sum() + (pooled * t["w_pooled"]).sum()).backward()       # two nodes on one pack, one pass
    named = dict(te.named_parameters())
    for k in ("module.embeddings.word_embeddings.weight", "module.embeddings.token_type_embeddings.weight",
              "module.encoder.layer.0.intermediate.dense.weight", "module.encoder.layer.1.output.dense.weight",
              "module.pooler.dense.weight"):
        assert rel(named[k].grad, t["grads"][k]) < 6e-2, k
    assert torch.count_nonzero(named["module.embeddings.word_embeddings.weight"].grad[0]) == 0


def test_mmft_backend_and_vilbert_image_embeddings_vs_reference_golden_cpu(cpu_frontends):
    from mmf_b200.registry import registry
    g = golden_io.load("mmft_embeddings")
    tcfg = types.SimpleNamespace(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=1,
                                 hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, layer_norm_eps=1e-12,
                                 hidden_act="gelu", initializer_range=0.02, vocab_size=50, max_position_embeddings=32,
                                 type_vocab_size=2, pad_token_id=0)
    mods = [dict(type="text", key="text", position_dim=32, embedding_dim=64, segment_id=0),
            dict(type="image", key="image", position_dim=16, embedding_dim=40, segment_id=1)]
    backend = registry.get_transformer_backend_class("b200")(
        dict(modalities=mods, transformer_config=tcfg, token_noise_mean=0.0, token_noise_std=0.01))
    backend.embeddings.load_state_dict(g["state_dict"])
    backend.eval()
    emb = backend.generate_embeddings(g["tokens"], g["pos"], g["seg"], None)
    assert rel(emb, g["out"]) < 2e-2
    assert torch.equal(backend.generate_attention_mask(list(g["masks"])), g["attention_mask"])
    seq, first = backend(g["tokens"], g["pos"], g["seg"], list(g["masks"]))
    assert seq.shape == (2, 11, 64) and torch.isfinite(seq.float()).all()
    ge = golden_io.load("embeddings")
    mod = cpu_frontends.VB.B200ImageFeatureEmbeddings(
        types.SimpleNamespace(v_feature_size=40, v_hidden_size=96, hidden_dropout_prob=0.1))
    mod.load_state_dict(ge["img_state_dict"])
    mod.eval()
    assert rel(mod(ge["feats"], ge["loc"]), ge["img_out"]) < 2e-2


def test_monkey_patch_swap_on_hf_bert_encoder_cpu(cpu_modules):
    """replace_with_b200() (the reference's replace_with_jit() boundary): a stock HuggingFace BertEncoder runs on the
    engine, keeps its parameter names, and the original forward is restored by undo."""
    from transformers import BertConfig
    from transformers.models.bert.modeling_bert import BertEncoder
    from mmf_b200.patch import replace_with_b200, undo_replace_with_b200
    torch.manual_seed(0)
    cfg = BertConfig(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=2, vocab_size=50,
                     hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    enc = BertEncoder(cfg).eval()
    keys = set(enc.state_dict().keys())
    x = torch.randn(2, 9, 64)
    mask = torch.ones(2, 9, dtype=torch.long)
    mask[0, 6:] = 0
    add = O.extended_attention_mask(mask)
    orig_forward = BertEncoder.forward
    replace_with_b200()
    try:
        out = enc(x, add)[0]
    finally:
        undo_replace_with_b200()
    assert BertEncoder.forward is orig_forward and set(enc.state_dict().keys()) == keys
    sd = {k: v.detach().to(torch.bfloat16).float() for k, v in enc.state_dict().items()}
    assert rel(out, O.bert_encoder(x.to(torch.bfloat16).float(), add, sd, "", 2, 1)) < 2e-2


def test_visual_bert_trunk_vs_oracle_cpu(cpu_frontends):
    """SampleList -> masks (integer, exact) -> embeddings -> encoder -> pooler, the bench's model at toy size"""
    from mmf_b200.visual_bert import B200VisualBERT
    cfg = types.SimpleNamespace(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=2,
                                vocab_size=50, max_position_embeddings=64, type_vocab_size=2, visual_embedding_dim=40,
                                hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, layer_norm_eps=1e-12,
                                hidden_act="gelu", initializer_range=0.02)
    torch.manual_seed(2)
    model = B200VisualBERT(cfg).eval()
    _bf16_round_(model)
    B, T, R = 3, 9, 5
    ids = torch.randint(1, 50, (B, T))
    imask = torch.ones(B, T, dtype=torch.long)
    imask[0, 6:] = 0
    seg = torch.zeros(B, T, dtype=torch.long)
    feats = torch.randn(B, R, 40).abs().to(torch.bfloat16).float()
    maxf = torch.tensor([5, 3, 4])
    out = model({"input_ids": ids, "input_mask": imask, "segment_ids": seg, "image_feature_0": feats,
                 "image_info_0": {"max_features": maxf}})
    image_mask, vtype, att = O.visual_bert_masks(imask, maxf, R)
    assert torch.equal(out["image_mask"], image_mask) and torch.equal(out["attention_mask"], att)
    sd = {k: v.detach() for k, v in model.bert.state_dict().items()}
    emb = O.visio_linguistic_embeddings(ids, seg, feats, vtype, sd, "embeddings")
    seq = O.bert_encoder(emb, O.extended_attention_mask(att), sd, "encoder", 2, 1)
    assert rel(out["sequence_output"], seq) < 2e-2
    assert rel(out["pooled_output"], O.bert_pooler(seq, sd, "pooler")) < 2e-2


def test_uniter_model_base_vs_reference_golden_cpu(cpu_frontends, monkeypatch):
    import mmf_b200.uniter as UN
    monkeypatch.setattr(UN, "_require_cuda", lambda t, what: None)
    g = golden_io.load("uniter")
    c = g["cfg"]
    cfg = types.SimpleNamespace(hidden_size=c["hidden"], num_attention_heads=c["heads"], intermediate_size=c["inter"],
                                num_hidden_layers=c["layers"], vocab_size=c["vocab"], max_position_embeddings=c["max_pos"],
                                type_vocab_size=2, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                                layer_norm_eps=1e-12, initializer_range=0.02)
    m = UN.B200UNITERModelBase(cfg, img_dim=c["img_dim"])
    ref_keys = {k for k in g["state_dict"] if not k.endswith("position_ids") and not k.endswith("token_type_ids")}
    assert set(m.state_dict().keys()) == ref_keys                   # HF's index buffers aside, the reference's names
    m.load_state_dict({k: v for k, v in g["state_dict"].items() if k in ref_keys})
    m.eval()
    feat = g["feat"].clone().requires_grad_(True)
    out = m(g["ids"], g["pos_ids"], feat, g["pos"], g["att"])
    assert len(out.hidden_layers) == g["n_hidden"]
    assert rel(out.final_layer, g["final"]) < 2e-2 and rel(out.hidden_layers[1], g["hidden_1"]) < 2e-2
    (out.final_layer * g["w_rand"]).sum().backward()
    assert rel(feat.grad, g["dfeat"]) < 4e-2
    named = dict(m.named_parameters())
    for k in ("img_embeddings.img_linear.weight", "img_embeddings.pos_linear.weight", "img_embeddings.final_layer_norm.weight",
              "img_embeddings.img_layer_norm.bias", "text_embeddings.token_type_embeddings.weight",
              "encoder.layer.1.intermediate.dense.weight"):
        assert rel(named[k].grad, g["grads"][k]) < 6e-2, k
    with torch.no_grad():
        masked = m(g["ids"], g["pos_ids"], g["feat"], g["pos"], g["att"], img_masks=g["img_masks"]).final_layer
        assert rel(masked, g["final_masked"]) < 2e-2
        T = g["ids"].shape[1]
        img_only = m(g["ids"], g["pos_ids"], g["feat"], g["pos"], g["att"][:, T:], input_modality="image").final_layer
        assert rel(img_only, g["final_image_only"]) < 2e-2
        # the reference passes position ids as [1, T] (uniter.py:732-737) and HF broadcasts them over the batch
        assert g["ids"].shape[0] > 1 and torch.equal(g["pos_ids"], g["pos_ids"][:1].expand_as(g["pos_ids"]))
        bc = m(g["ids"], g["pos_ids"][:1], g["feat"], g["pos"], g["att"]).final_layer
        assert torch.equal(bc, m(g["ids"], g["pos_ids"], g["feat"], g["pos"], g["att"]).final_layer)


def test_lxmert_encoder_vs_reference_golden_cpu(cpu_frontends, monkeypatch):
    """language / relational layers + cross-modality layers whose ONE cross-attention block serves both directions:
    its weight gradients are the sum of the two uses (engine.xlayer_bwd accumulates both into the same regions)."""
    import mmf_b200.lxmert as LX
    monkeypatch.setattr(LX, "_require_cuda", lambda t, what: None)
    g = golden_io.load("lxmert")
    c = g["cfg"]
    cfg = types.SimpleNamespace(hidden_size=c["hidden"], num_attention_heads=c["heads"], intermediate_size=c["inter"],
                                hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, visual_feat_dim=c["feat_dim"],
                                visual_pos_dim=c["pos_dim"], l_layers=c["l"], x_layers=c["x"], r_layers=c["r"])
    enc = LX.B200LXMERTEncoder(cfg)
    assert set(enc.state_dict().keys()) == set(g["state_dict"].keys())
    enc.load_state_dict(g["state_dict"])
    enc.eval()
    lang = g["lang"].clone().requires_grad_(True)
    feats = g["feats"].clone().requires_grad_(True)
    lo, vo = enc(lang, O.extended_attention_mask(g["lmask"]), (feats, g["boxes"]), O.extended_attention_mask(g["vmask"]))
    assert rel(lo, g["lang_out"]) < 2e-2 and rel(vo, g["visn_out"]) < 2e-2
    ((lo * g["wl"]).sum() + (vo * g["wv"]).sum()).backward()
    assert rel(lang.grad, g["dlang"]) < 4e-2 and rel(feats.grad, g["dfeats"]) < 4e-2
    for n, p in enc.named_parameters():
        if "key" in n and n.endswith("bias"):
            continue
        assert rel(p.grad, g["grads"][n]) < 8e-2, n


def test_masked_lm_head_vs_reference_golden_cpu(cpu_frontends, monkeypatch):
    """vocabulary 203 (not a multiple of 8): padded compute copy of the tied decoder weight, logits = column slice;
    loss over all positions == loss over the labelled rows only"""
    import mmf_b200.heads as HD
    monkeypatch.setattr(HD, "_require_cuda", lambda t, what: None)
    g = golden_io.load("mlm_head")
    cfg = types.SimpleNamespace(hidden_size=g["cfg"]["hidden"], vocab_size=g["cfg"]["vocab"], layer_norm_eps=1e-12,
                                initializer_range=0.02)
    emb = torch.nn.Embedding(cfg.vocab_size, cfg.hidden_size)
    cls = HD.B200BertPreTrainingHeads(cfg, emb.weight)
    assert cls.predictions.decoder.weight is emb.weight and cls.predictions.decoder.bias is cls.predictions.bias
    keys = set(cls.state_dict().keys())
    assert {"predictions.bias", "predictions.decoder.bias", "predictions.decoder.weight",
            "predictions.transform.dense.weight", "predictions.transform.LayerNorm.bias", "seq_relationship.weight"} <= keys
    sd = {k[len("cls."):]: v for k, v in g["state_dict"].items()}
    sd["predictions.decoder.bias"] = sd["predictions.bias"]
    cls.load_state_dict(sd)
    cls.eval()
    seq = g["seq"].clone().requires_grad_(True)
    scores, rel_score = cls(seq, g["pooled"])
    assert scores.shape == g["scores"].shape and rel(scores, g["scores"]) < 2e-2 and rel(rel_score, g["rel"]) < 1e-5
    loss, logits = HD.masked_lm_loss(cls, seq, g["labels"])
    assert abs(loss.item() - g["loss"].item()) < 2e-2 * abs(g["loss"].item())
    loss.backward()
    assert rel(seq.grad, g["dseq"]) < 5e-2
    named = dict(cls.named_parameters())
    for k in ("predictions.transform.dense.weight", "predictions.transform.LayerNorm.weight", "predictions.decoder.weight",
              "predictions.bias"):
        assert rel(named[k].grad, g["grads"]["cls." + k]) < 6e-2, k
    assert emb.weight.grad is named["predictions.decoder.weight"].grad        # the tie: one parameter, one gradient
    full = loss.item()
    cls.zero_grad(set_to_none=True)
    loss_m, logits_m = HD.masked_lm_loss(cls, seq.detach(), g["labels"], positions="masked")
    assert logits_m.shape == (4, cfg.vocab_size) and abs(loss_m.item() - full) < 1e-3 * abs(full)
    # positions="fused": gather -> transform -> chunked (vocabulary GEMM -> loss kernel writing d(logits) in place -> dgrad /
    # wgrad): same loss and gradients as the reference's materialised logits, no logits tensor
    cls.zero_grad(set_to_none=True)
    seq2 = g["seq"].clone().requires_grad_(True)
    loss_f, none = HD.masked_lm_loss(cls, seq2, g["labels"], positions="fused")
    assert none is None and abs(loss_f.item() - g["loss"].item()) < 2e-2 * abs(g["loss"].item())
    (loss_f * 1.5).backward()                       # a non-unit incoming gradient scales the precomputed gradients
    assert rel(seq2.grad, 1.5 * g["dseq"]) < 5e-2
    for k in ("predictions.transform.dense.weight", "predictions.transform.LayerNorm.weight", "predictions.decoder.weight",
              "predictions.bias"):
        assert rel(named[k].grad, 1.5 * g["grads"]["cls." + k]) < 6e-2, k
    # chunking does not change the result
    import mmf_b200.ops as OPS
    hh = torch.randn(37, 64).to(torch.bfloat16).float()
    ww = (torch.randn(203, 64) * 0.1).requires_grad_(True)
    bbias = (torch.randn(203) * 0.1).requires_grad_(True)
    lab = torch.randint(0, 203, (37,))
    lab[::5] = -1
    ref = torch.nn.functional.cross_entropy(torch.nn.functional.linear(hh, ww.to(torch.bfloat16).float(), bbias.to(torch.bfloat16).float()),
                                            lab, ignore_index=-1)
    for chunk in (8, 37, 1000):
        ww.grad = bbias.grad = None
        lf = OPS.linear_cross_entropy(hh, ww, bbias, lab, -1, chunk_rows=chunk)
        assert abs(lf.item() - ref.item()) < 2e-2 * abs(ref.item()), chunk
        lf.backward()
        assert ww.grad.shape == ww.shape and torch.isfinite(ww.grad).all() and bbias.grad.abs().sum() > 0


def test_visual_bert_for_pretraining_vs_oracle_cpu(cpu_frontends, monkeypatch):
    """visual_bert/pretrain (BASELINE.json configs[1]) end to end: trunk + tied MLM head + loss and its gradients"""
    import mmf_b200.heads as HD
    from mmf_b200.visual_bert import B200VisualBERTForPretraining
    monkeypatch.setattr(HD, "_require_cuda", lambda t, what: None)
    cfg = types.SimpleNamespace(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=2,
                                vocab_size=51, max_position_embeddings=64, type_vocab_size=2, visual_embedding_dim=40,
                                hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, layer_norm_eps=1e-12,
                                hidden_act="gelu", initializer_range=0.02)
    torch.manual_seed(4)
    model = B200VisualBERTForPretraining(cfg).eval()
    _bf16_round_(model)
    B, T, R = 2, 8, 4
    ids = torch.randint(1, 51, (B, T))
    seg = torch.zeros(B, T, dtype=torch.long)
    feats = torch.randn(B, R, 40).abs().to(torch.bfloat16).float()
    vtype = torch.zeros(B, R, dtype=torch.long)
    att = torch.ones(B, T + R, dtype=torch.long)
    att[1, 6:T] = 0
    labels = torch.full((B, T + R), -1, dtype=torch.long)
    labels[0, 1], labels[0, 4], labels[1, 2] = 7, 50, 19
    out = model(ids, None, att, seg, feats, vtype, masked_lm_labels=labels)
    assert out["logits"].shape == (B, T + R, 51) and out["loss"] is out["masked_lm_loss"]
    out["loss"].backward()
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in model.state_dict().items()}
    sd["cls.predictions.decoder.weight"] = sd["bert.embeddings.word_embeddings.weight"]        # the tie
    emb = O.visio_linguistic_embeddings(ids, seg, feats, vtype, sd, "bert.embeddings")
    seq = O.bert_encoder(emb, O.extended_attention_mask(att), sd, "bert.encoder", 2, 1)
    scores, _ = O.bert_pretraining_heads(seq, O.bert_pooler(seq, sd, "bert.pooler"), sd, "cls")
    loss = O.masked_lm_loss(scores, labels)
    loss.backward()
    assert abs(out["loss"].item() - loss.item()) < 2e-2 * abs(loss.item())
    assert rel(out["logits"], scores) < 2e-2
    named = dict(model.named_parameters())
    for k in ("bert.embeddings.word_embeddings.weight", "bert.encoder.layer.1.output.dense.weight",
              "cls.predictions.transform.dense.weight", "bert.embeddings.projection.weight"):
        assert rel(named[k].grad, sd[k].grad) < 8e-2, k


def test_visual_bert_bypass_transformer_vs_reference_golden_cpu(cpu_frontends):
    from mmf_b200.visual_bert import B200VisualBERTBase
    g = golden_io.load("visual_bert_bypass")
    c = g["cfg"]
    cfg = types.SimpleNamespace(hidden_size=c["hidden"], num_attention_heads=c["heads"], intermediate_size=c["inter"],
                                num_hidden_layers=c["layers"], vocab_size=c["vocab"], max_position_embeddings=c["max_pos"],
                                type_vocab_size=2, visual_embedding_dim=c["vdim"], hidden_dropout_prob=0.0,
                                attention_probs_dropout_prob=0.0, layer_norm_eps=1e-12, hidden_act="gelu",
                                initializer_range=0.02, bypass_transformer=True)
    m = B200VisualBERTBase(cfg)
    ref_keys = {k for k in g["state_dict"] if not k.endswith("position_ids") and not k.endswith("token_type_ids")}
    assert set(m.state_dict().keys()) == ref_keys
    m.load_state_dict({k: v for k, v in g["state_dict"].items() if k in ref_keys})
    m.eval()
    feats = g["feats"].clone().requires_grad_(True)
    seq, pooled, _ = m(g["ids"], g["att"], g["seg"], feats, g["vtype"])
    assert rel(seq, g["seq"]) < 2e-2 and rel(pooled, g["pooled"]) < 2e-2
    (seq * g["w_rand"]).sum().backward()
    assert rel(feats.grad, g["dfeats"]) < 4e-2
    named = dict(m.named_parameters())
    for k in ("additional_layer.attention.self.query.weight", "additional_layer.output.dense.weight",
              "encoder.layer.1.intermediate.dense.weight", "embeddings.projection.weight",
              "embeddings.word_embeddings.weight"):
        assert rel(named[k].grad, g["grads"][k]) < 6e-2, k
    m.bypass_transformer = False
    with torch.no_grad():
        ps, pp, _ = m(g["ids"], g["att"], g["seg"], g["feats"], g["vtype"])
    assert rel(ps, g["plain_seq"]) < 2e-2 and rel(pp, g["plain_pooled"]) < 2e-2


def test_vilbert_base_front_to_back_vs_oracle_cpu(cpu_frontends):
    """ids / region features / locations -> text + image embeddings -> two-stream encoder -> poolers"""
    c = dict(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=2, vocab_size=50,
             max_position_embeddings=32, type_vocab_size=2, v_feature_size=40, v_hidden_size=128, v_num_attention_heads=2,
             v_intermediate_size=128, v_num_hidden_layers=1, bi_hidden_size=128, bi_num_attention_heads=2,
             v_biattention_id=[0], t_biattention_id=[1])
    cfg = types.SimpleNamespace(hidden_dropout_prob=0.0, v_hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                                v_attention_probs_dropout_prob=0.0, layer_norm_eps=1e-12, initializer_range=0.02, **c)
    torch.manual_seed(6)
    m = cpu_frontends.VB.B200ViLBERTBase(cfg).eval()
    _bf16_round_(m)
    B, T, R = 2, 7, 5
    ids = torch.randint(1, 50, (B, T))
    feats = torch.randn(B, R, 40).to(torch.bfloat16).float()
    loc = torch.rand(B, R, 5).to(torch.bfloat16).float()
    tmask = torch.ones(B, T, dtype=torch.long)
    tmask[0, 5:] = 0
    imask = torch.ones(B, R, dtype=torch.long)
    imask[1, 3:] = 0
    out = m(ids, feats, loc, attention_mask=tmask, image_attention_mask=imask, reference_outputs=True)
    assert len(out) == 7 and out[4] is None and out[5] is None
    sd = {k: v.detach() for k, v in m.state_dict().items()}
    temb = O.bert_embeddings(ids, torch.zeros_like(ids), sd, "embeddings")
    vemb = O.image_feature_embeddings(feats, loc, sd, "v_embeddings")
    t_out, v_out = O.vilbert_encoder(temb, vemb, O.extended_attention_mask(tmask), O.extended_attention_mask(imask),
                                     {k[len("encoder."):]: v for k, v in sd.items() if k.startswith("encoder.")}, "", c)
    assert rel(out[0], t_out) < 2e-2 and rel(out[1], v_out) < 2e-2
    pt = torch.relu(t_out[:, 0] @ sd["t_pooler.dense.weight"].t() + sd["t_pooler.dense.bias"])
    pv = torch.relu(v_out[:, 0] @ sd["v_pooler.dense.weight"].t() + sd["v_pooler.dense.bias"])
    assert rel(out[2], pt) < 3e-2 and rel(out[3], pv) < 3e-2
    seq_t, seq_v, _ = m(ids, feats, loc, attention_mask=tmask, image_attention_mask=imask)      # default: trunk outputs only
    assert torch.equal(seq_t, out[0]) and torch.equal(seq_v, out[1])


def test_vit_model_vs_reference_golden_cpu(cpu_frontends, monkeypatch):
    """pre-LN (ViT) layer = the post-LN layer's kernels in a different order (engine.vit_layer_fwd / _bwd): encoder with a
    key-padding mask (forward, hidden states, input and parameter gradients) and the model tail from pixels (patch
    projection as a GEMM over unfolded patches, [CLS] + position table, final LayerNorm, pooler) vs mmf/modules/vit.py"""
    import mmf_b200.vit as VT
    monkeypatch.setattr(VT, "_require_cuda", lambda t, what: None)
    g = golden_io.load("vit")
    c = g["cfg"]
    cfg = types.SimpleNamespace(hidden_size=c["hidden"], num_attention_heads=c["heads"], intermediate_size=c["inter"],
                                num_hidden_layers=c["layers"], hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                                layer_norm_eps=1e-12, hidden_act="gelu", image_size=c["image_size"], patch_size=c["patch_size"],
                                num_channels=3, initializer_range=0.02)
    m = VT.B200ViTModel(cfg)
    assert set(m.state_dict().keys()) == set(g["state_dict"].keys())          # HF ViT / reference parameter names
    m.load_state_dict(g["state_dict"])
    m.eval()
    x = g["x"].clone().requires_grad_(True)
    add = O.extended_attention_mask(g["mask"])
    out = m.encoder(x, attention_mask=add, output_hidden_states=True, return_dict=False)
    assert len(out[1]) == g["n_hidden"]
    assert rel(out[0], g["out"]) < 2e-2 and rel(out[1][1], g["hidden_1"]) < 2e-2
    (out[0] * g["w_rand"]).sum().backward()
    assert rel(x.grad, g["dx"]) < 3e-2
    named = dict(m.named_parameters())
    for k, gr in g["grads"].items():
        if "key.bias" in k:
            continue
        assert rel(named[k].grad, gr) < 8e-2, k
    with torch.no_grad():
        seq, pooled = m(g["pixels"])
        assert rel(m.embeddings(g["pixels"]), g["embedded"]) < 2e-2
        assert rel(seq, g["seq_from_pixels"]) < 2e-2 and rel(pooled, g["pooled_from_pixels"]) < 2e-2
    # train mode with dropout: the masks reach the backward through mmfb_dropout_apply; repeatable under manual_seed
    cfg.hidden_dropout_prob = cfg.attention_probs_dropout_prob = 0.1
    enc = VT.B200ViTEncoder(cfg).train()
    xx = torch.randn(2, 9, c["hidden"])

    def run():
        torch.manual_seed(3)
        cpu_frontends_seed_reset()
        xi = xx.clone().requires_grad_(True)
        o = enc(xi, return_dict=False)[0]
        o.square().sum().backward()
        return o.detach().clone(), xi.grad.clone()
    import mmf_b200.modules as MM

    def cpu_frontends_seed_reset():
        MM._SEED_COUNTER[0] = 0
    (o1, g1), (o2, g2) = run(), run()
    assert torch.equal(o1, o2) and torch.equal(g1, g2) and torch.isfinite(g1).all()


def test_vinvl_base_vs_reference_golden_cpu(cpu_frontends, monkeypatch):
    import mmf_b200.vinvl as VV
    monkeypatch.setattr(VV, "_require_cuda", lambda t, what: None)
    g = golden_io.load("vinvl")
    c = g["cfg"]
    cfg = types.SimpleNamespace(hidden_size=c["hidden"], num_attention_heads=c["heads"], intermediate_size=c["inter"],
                                num_hidden_layers=c["layers"], vocab_size=c["vocab"], max_position_embeddings=c["max_pos"],
                                type_vocab_size=2, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                                layer_norm_eps=1e-12, initializer_range=0.02, img_feature_dim=c["img_dim"],
                                use_img_layernorm=True, img_layer_norm_eps=1e-12)
    m = VV.B200VinVLBase(cfg)
    assert set(m.state_dict().keys()) == set(g["state_dict"].keys())
    m.load_state_dict(g["state_dict"])
    m.eval()
    feats = g["feats"].clone().requires_grad_(True)
    out = m(g["ids"], feats, attention_mask=g["att"])
    assert len(out.hidden_layers) == g["n_hidden"]
    assert rel(out.last_hidden_state, g["last"]) < 2e-2 and rel(out.hidden_layers[1], g["hidden_1"]) < 2e-2
    (out.last_hidden_state * g["w_rand"]).sum().backward()
    assert rel(feats.grad, g["dfeats"]) < 4e-2
    named = dict(m.named_parameters())
    for k in ("img_embedding.0.weight", "img_embedding.1.weight", "embeddings.word_embeddings.weight",
              "encoder.layer.1.output.dense.weight"):
        assert rel(named[k].grad, g["grads"][k]) < 8e-2, k
    with pytest.raises(NotImplementedError):
        m(g["ids"], g["feats"], attention_mask=torch.ones(3, 12, 12))
