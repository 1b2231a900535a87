"""CPU tests of the host-side logic (no GPU compute): C-ABI export, parameter pack, schedules, key names."""
import ctypes
import types

import pytest
import torch

from oracle import golden_io


def test_library_loads_and_exports_every_declared_symbol():
    from mmf_b200 import lib
    syms = lib.header_symbols()
    assert len(syms) >= 10
    for s in syms:
        assert hasattr(lib.LIB, s), s
    assert lib.LIB.mmfb_version() >= 100


def test_compute_entry_points_fail_loudly_without_gpu():
    from mmf_b200 import lib
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    a = lib.GemmArgs()
    rc = lib.LIB.mmfb_gemm(ctypes.byref(a), None)
    assert rc == lib.MMFB_ERR_DEVICE
    assert "no CPU fallback" in lib.last_error()
    with pytest.raises(RuntimeError):
        lib.check(rc)


def test_param_pack_views_and_grad_handover():
    from mmf_b200.engine import ParamPack
    lin = [torch.nn.Linear(8, 16), torch.nn.Linear(8, 16), torch.nn.Linear(8, 16)]
    params = [l.weight for l in lin] + [l.bias for l in lin]
    before = [p.detach().clone() for p in params]
    pack = ParamPack(params, "cpu")
    for p, b in zip(params, before):
        assert torch.equal(p.detach(), b)
    assert pack.intact()
    h = pack.handle(*params[0:3])           # fused q/k/v weight
    assert tuple(h.w.shape) == (48, 8) and tuple(h.g.shape) == (48, 8)
    # optimizer-style in-place update lands in the master buffer
    with torch.no_grad():
        params[1].add_(1.0)
    assert torch.equal(pack.master[pack.offsets[1]:pack.offsets[1] + 128].view(16, 8), params[1].detach())
    aliased = pack.prepare_grads()
    assert not any(aliased)
    grads = pack.autograd_grads(aliased)
    for p, g in zip(params, grads):
        p.grad = g
    assert all(pack.prepare_grads())        # now aliased -> accumulate in place, autograd gets None
    assert all(g is None for g in pack.autograd_grads([True] * len(params)))
    lin[0].weight.data = lin[0].weight.data.clone()
    assert not pack.intact()
    with pytest.raises(ValueError):
        pack.handle(params[0], params[2])   # not adjacent


def test_param_pack_two_nodes_in_one_backward_pass():
    # the same pack behind two autograd nodes of one graph (an encoder applied twice before a single backward):
    # the second node must accumulate into the flat buffer instead of zeroing the first node's result
    from mmf_b200.engine import ParamPack
    w = torch.nn.Parameter(torch.randn(16, 8))
    pack = ParamPack([w], "cpu")

    class Scale(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x, w_):
            ctx.save_for_backward(x)
            return x @ w_.detach().t()

        @staticmethod
        def backward(ctx, dy):
            (x,) = ctx.saved_tensors
            aliased = pack.prepare_grads()
            pack.grad_view(w).add_(dy.t() @ x)            # kernels accumulate into the flat buffer
            return dy @ w.detach(), pack.autograd_grads(aliased)[0]

    x1, x2 = torch.randn(4, 8), torch.randn(4, 8)
    (Scale.apply(x1, w).sum() + 3.0 * Scale.apply(x2, w).sum()).backward()
    expect = torch.ones(4, 16).t() @ x1 + 3.0 * torch.ones(4, 16).t() @ x2
    assert torch.allclose(w.grad, expect, atol=1e-5)
    assert w.grad.data_ptr() == pack.grad.data_ptr()        # adopted without a copy
    # next pass, gradient accumulation (p.grad kept) and then zero_grad(set_to_none)
    Scale.apply(x1, w).sum().backward()
    assert torch.allclose(w.grad, expect + torch.ones(4, 16).t() @ x1, atol=1e-5)
    w.grad = None
    Scale.apply(x2, w).sum().backward()
    assert torch.allclose(w.grad, torch.ones(4, 16).t() @ x2, atol=1e-5)


def test_vilbert_schedule_matches_oracle():
    from mmf_b200.modules import vilbert_schedule
    from oracle.fusion_oracle import vilbert_schedule as oracle_schedule
    args = ([0, 1, 2, 3, 4, 5], [6, 7, 8, 9, 10, 11], 12, 6)
    assert vilbert_schedule(*args) == oracle_schedule(*args)
    assert vilbert_schedule([0, 1], [1, 2], 3, 2) == oracle_schedule([0, 1], [1, 2], 3, 2)


def test_state_dict_keys_match_reference_modules():
    from mmf_b200.modules import B200BertEncoder, B200ViLBertEncoder
    g = golden_io.load("bert_encoder")
    c = g["cfg"]
    cfg = types.SimpleNamespace(hidden_size=c["hidden"], num_attention_heads=c["heads"], intermediate_size=c["inter"],
                                num_hidden_layers=c["layers"], hidden_dropout_prob=0.1,
                                attention_probs_dropout_prob=0.1, layer_norm_eps=1e-12)
    enc = B200BertEncoder(cfg)
    assert {k: tuple(v.shape) for k, v in enc.state_dict().items()} == {k: tuple(v.shape) for k, v in
                                                                        g["state_dict"].items()}
    g = golden_io.load("vilbert_encoder")
    cfg = types.SimpleNamespace(hidden_dropout_prob=0.1, v_hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1,
                                v_attention_probs_dropout_prob=0.1, **g["cfg"])
    enc = B200ViLBertEncoder(cfg)
    assert {k: tuple(v.shape) for k, v in enc.state_dict().items()} == {k: tuple(v.shape) for k, v in
                                                                        g["state_dict"].items()}


def test_bad_head_split_raises_like_reference():
    from mmf_b200.modules import B200BertEncoder
    cfg = types.SimpleNamespace(hidden_size=100, num_attention_heads=3, intermediate_size=64, num_hidden_layers=1,
                                hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, layer_norm_eps=1e-12)
    with pytest.raises(ValueError):
        B200BertEncoder(cfg)


def test_best_splits_prefers_full_waves():
    from mmf_b200.engine import best_splits
    assert best_splits(768, 768, 14592) >= 4      # 18 tiles -> needs split-K to fill 148 SMs
    assert best_splits(3072, 768, 14592) >= 2
    assert best_splits(128, 256, 64) == 1         # a single k-block cannot be split


def test_additive_mask_shapes():
    from mmf_b200.engine import additive_mask_2d
    m4 = torch.zeros(2, 1, 1, 5)
    assert tuple(additive_mask_2d(m4, 2, 5).shape) == (2, 5)
    assert additive_mask_2d(None, 2, 5) is None
    with pytest.raises(ValueError):
        additive_mask_2d(torch.zeros(2, 1, 5, 5), 2, 5)


def test_registry_and_sample_list_shims():
    from mmf_b200.registry import registry
    from mmf_b200.sample import SampleList
    import mmf_b200.mmft_backend  # noqa: F401  (registers "b200")
    assert registry.get_transformer_backend_class("b200").__name__ == "B200TransformerBackend"
    assert registry.get_transformer_backend_class("nope") is None
    sl = SampleList()
    sl.input_ids = torch.zeros(3, 4, dtype=torch.long)
    sl["image_info_0"] = {"max_features": torch.tensor([1, 2, 3])}
    assert sl.get_batch_size() == 3 and sl.fields() == ["input_ids", "image_info_0"]
    moved = sl.to("cpu")
    assert torch.equal(moved.image_info_0["max_features"], torch.tensor([1, 2, 3]))
    with pytest.raises(AttributeError):
        sl.missing


def test_encoder_plugins_registered_with_reference_names_and_keys():
    # mmf/modules/encoders.py:116,183,513 register these names; state-dict keys are the reference's
    import mmf_b200.encoders as enc
    from mmf_b200.registry import registry
    assert registry.get_encoder_class("finetune_faster_rcnn_fpn_fc7") is enc.B200FinetuneFasterRcnnFpnFc7
    assert registry.get_encoder_class("identity") is enc.B200IdentityEncoder
    assert registry.get_encoder_class("transformer") is enc.B200TransformerEncoder
    g = golden_io.load("encoders")
    c = g["transformer"]["cfg"]
    te = enc.B200TransformerEncoder(dict(hidden_size=c["hidden"], num_hidden_layers=c["layers"],
                                         num_attention_heads=c["heads"], intermediate_size=c["inter"],
                                         vocab_size=c["vocab"], max_position_embeddings=c["max_pos"],
                                         num_segments=c["num_segments"]))
    assert set(te.state_dict().keys()) == set(g["transformer"]["state_dict"].keys())
    assert te.embeddings is te.module.embeddings
    fc7 = enc.B200FinetuneFasterRcnnFpnFc7({"in_dim": 256, "out_dim": 128})
    assert set(fc7.state_dict().keys()) == set(g["fc7"]["state_dict"].keys())
    ident = enc.B200IdentityEncoder({"in_dim": 64})
    x = torch.randn(2, 64)
    assert ident(x) is x and ident.out_dim == 64
    with pytest.raises(RuntimeError):      # no CPU fallback
        fc7(torch.randn(2, 256))


def test_encoder_factories_and_mmbt_construction_route():
    # build_encoder / factories / MultiModalEncoderBase (mmf/utils/build.py:495-546, encoders.py:79-113,454-485,588-646)
    import mmf_b200.encoders as enc
    from mmf_b200.mmbt import B200MMBTBase
    assert isinstance(enc.build_encoder({"type": "identity", "params": {"in_dim": 256}}), enc.B200IdentityEncoder)
    fc7 = enc.build_encoder({"type": "finetune_faster_rcnn_fpn_fc7", "params": {"in_dim": 64, "out_dim": 32}})
    assert isinstance(fc7, enc.B200FinetuneFasterRcnnFpnFc7) and fc7.out_dim == 32
    with pytest.raises(KeyError):
        enc.build_encoder({"type": "resnet152", "params": {}})
    f = enc.B200ImageFeatureEncoderFactory({"type": "default", "params": {"in_dim": 2048}})
    assert isinstance(f.module, torch.nn.Identity) and f.out_dim == 2048
    assert enc.B200ImageFeatureEncoderFactory({"type": "projection", "params": {"in_dim": 64, "out_dim": 16}}).out_dim == 16
    with pytest.raises(AssertionError):
        enc.B200ImageFeatureEncoderFactory({"type": "default", "params": {}})
    with pytest.raises(NotImplementedError):
        enc.B200ImageFeatureEncoderFactory({"type": "spatial", "params": {"in_dim": 4}})
    with pytest.raises(NotImplementedError):
        enc.build_image_encoder({"type": "resnet152", "params": {}}, direct_features=False)
    te_params = dict(hidden_size=128, num_hidden_layers=1, num_attention_heads=2, vocab_size=50,
                     max_position_embeddings=160, num_segments=2)
    cfg = dict(direct_features_input=True, modal_hidden_size=64, num_labels=2,
               text_encoder=dict(type="transformer", params=te_params),
               modal_encoder=dict(type="finetune_faster_rcnn_fpn_fc7", params=dict(in_dim=64, out_dim=64)))
    base = enc.B200MultiModalEncoderBase(cfg)
    assert base.encoder_config.hidden_size == 128 and base.modal_hidden_size == 64
    assert isinstance(base.modal_encoder, enc.B200FinetuneFasterRcnnFpnFc7)
    m = B200MMBTBase.from_config(cfg)
    keys = set(m.state_dict().keys())
    # the reference's key layout: MMBTModel.{transformer, modal_encoder.{encoder, proj_embeddings, shared tables}}
    for k in ("mmbt.modal_encoder.encoder.lc.weight", "mmbt.modal_encoder.proj_embeddings.weight",
              "mmbt.transformer.embeddings.word_embeddings.weight", "mmbt.transformer.pooler.dense.weight",
              "mmbt.transformer.encoder.layer.0.attention.self.query.weight", "mmbt.modal_encoder.word_embeddings.weight"):
        assert k in keys, k
    assert m.mmbt.modal_encoder.word_embeddings is m.mmbt.transformer.embeddings.word_embeddings
    assert m.mmbt.modal_encoder.proj_embeddings.in_features == 64 and m.num_max_segment == 2


def test_patch_and_undo_restore_forward():
    from transformers.models.bert.modeling_bert import BertEncoder
    from mmf_b200.patch import replace_with_b200, undo_replace_with_b200
    orig = BertEncoder.forward
    replace_with_b200()
    assert BertEncoder.forward is not orig
    undo_replace_with_b200()
    assert BertEncoder.forward is orig


def test_mmbt_token_surgery_matches_reference_golden_cpu():
    """integer path of MMBTBase.extract_modal_end_token is pure torch integer code: bit-exact on CPU too"""
    from mmf_b200.mmbt import extract_modal_end_token
    g = golden_io.load("mmbt")
    sl = {"input_ids": g["ids"].clone(), "input_mask": g["mask"].clone()}
    end = extract_modal_end_token(sl)
    assert torch.equal(end, g["end_token"])
    assert torch.equal(sl["input_ids"], g["shifted_ids"]) and torch.equal(sl["input_mask"], g["shifted_mask"])
