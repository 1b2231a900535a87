"""Model plugins (mmf_b200.models: registered `visual_bert` / `vilbert` / `mmbt`, SURVEY.md 8b 4th boundary form) on the CPU:
the host code (config handling, SampleList plumbing with its integer tensors, heads, loss wiring) runs over the kernel
test double (tests/fake_kernels.py) and is held to tests/golden/models.*.pt - outputs of the REFERENCE's own registered model
classes (oracle/make_golden.py::golden_models).  The kernels themselves are covered on the GPU (tests/test_models_gpu.py)."""
import os
import sys
import types

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import fake_kernels as FK  # noqa: E402
from oracle import golden_io  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


@pytest.fixture()
def cpu_models(monkeypatch):
    import mmf_b200.embeddings as EM
    import mmf_b200.encoders as EN
    import mmf_b200.engine as E
    import mmf_b200.heads as HD
    import mmf_b200.mmbt as MB
    import mmf_b200.modules as M
    import mmf_b200.ops as OPS
    import mmf_b200.vilbert as VB
    monkeypatch.setattr(E, "F", FK)
    monkeypatch.setattr(OPS, "F", FK)
    monkeypatch.setattr(EM, "F", FK)
    for mod in (M, EM, EN, MB, VB, HD):
        if hasattr(mod, "_require_cuda"):
            monkeypatch.setattr(mod, "_require_cuda", lambda t, what: None)
    import mmf_b200.models as MD
    return MD


def _sample_list(g, extra=None):
    from mmf_b200.sample import SampleList
    i = g["visual_bert_inputs"]
    sl = SampleList(input_ids=i["ids"].clone(), input_mask=i["mask"].clone(), segment_ids=i["seg"].clone(),
                    image_feature_0=i["feats"].clone(), image_info_0={"max_features": i["max_features"].clone()},
                    lm_label_ids=i["lm_label_ids"].clone(), targets=i["targets"].clone(), dataset_name="golden",
                    dataset_type="train")
    if extra:
        sl.update(extra)
    return sl


def _load(model, golden_sd):
    ours = model.state_dict()
    # HF <= 4.10 registers `position_ids` buffers and the pinned LM head keeps a `decoder.bias` alias: names aside from
    # those, the key sets are the reference's
    ref_keys = {k for k in golden_sd if not k.endswith("position_ids") and not k.endswith("token_type_ids")}
    assert set(ours.keys()) - {k for k in ours if k.endswith("decoder.bias")} == ref_keys - {k for k in ref_keys if k.endswith("decoder.bias")}
    model.load_state_dict({k: v for k, v in golden_sd.items() if k in ours})


@pytest.mark.parametrize("case", ["visual_bert_classification_default", "visual_bert_classification_vqa",
                                  "visual_bert_pretraining_default"])
def test_visual_bert_registered_model_vs_reference(cpu_models, case):
    MD = cpu_models
    g = golden_io.load("models")
    c = g[case]
    cfg = MD.load_model_config("visual_bert", overrides={k: v for k, v in c["config"].items()})
    cfg.losses = [{"type": "cross_entropy"}]
    assert MD.registry.get_model_class("visual_bert") is MD.VisualBERT
    assert MD.VisualBERT.config_path() == "configs/models/visual_bert/pretrain.yaml"
    model = MD.build_model(cfg).eval()
    _load(model, c["state_dict"])
    sl = _sample_list(g)
    out = model(sl)
    # integer paths: bit-exact
    assert torch.equal(sl["image_mask"], c["image_mask"]) and torch.equal(sl["attention_mask"], c["attention_mask"])
    if c["masked_lm_labels"] is not None:
        assert torch.equal(sl["masked_lm_labels"], c["masked_lm_labels"])
    if c["scores"] is not None:
        assert rel(out["scores"], c["scores"]) < 3e-2
        key = "train/golden/cross_entropy"
        assert list(out["losses"].keys()) == [key]                    # BaseModel.__call__ -> Losses (losses.py:209-212)
        loss = out["losses"][key].sum()
    else:
        assert sorted(out["losses"].keys()) == c["loss_keys"]
        assert rel(out["logits"], c["logits"]) < 3e-2
        loss = out["losses"]["golden/train/masked_lm_loss"]
    assert abs(float(loss) - float(c["loss"])) < 2e-2 * max(1.0, abs(float(c["loss"])))
    loss.backward()
    named = dict(model.named_parameters())
    checked = 0
    for k, gr in c["grads"].items():
        if k in named and named[k].grad is not None and gr.norm() > 1e-6 and any(
                s in k for s in ("classifier", "layer.1.output.dense.weight", "projection.weight", "cls.predictions.transform")):
            assert rel(named[k].grad, gr) < 8e-2, k
            checked += 1
    assert checked >= 3


@pytest.mark.parametrize("head", ["classification", "pretraining"])
def test_vilbert_registered_model_vs_reference(cpu_models, head):
    MD = cpu_models
    g = golden_io.load("models")
    c = g["vilbert_" + head]
    cfg = MD.load_model_config("vilbert", overrides=dict(c["config"]))
    cfg.losses = [{"type": "cross_entropy"}]
    model = MD.build_model(cfg).eval()
    _load(model, c["state_dict"])
    v = g["vilbert_inputs"]
    sl = _sample_list(g, {"image_labels": v["image_labels"].clone()})
    sl["image_info_0"] = {"max_features": g["visual_bert_inputs"]["max_features"].clone(), "bbox": v["bbox"].clone(),
                          "cls_prob": v["cls_prob"].numpy().copy()}
    out = model(sl)
    if head == "classification":
        assert rel(out["scores"], c["scores"]) < 3e-2
        loss = out["losses"]["train/golden/cross_entropy"].sum()
    else:
        assert sorted(out["losses"].keys()) == sorted(c["losses"].keys())
        for k in c["losses"]:
            assert abs(float(out["losses"][k]) - float(c["losses"][k])) < 3e-2 * max(1.0, abs(float(c["losses"][k]))), k
        loss = sum(x.sum() for x in out["losses"].values())
    assert abs(float(loss) - float(c["loss"])) < 3e-2 * max(1.0, abs(float(c["loss"])))
    loss.backward()
    named = dict(model.named_parameters())
    # the reference's never-used q_dense* stay without gradient here too
    for k in c["unused"]:
        if "q_dense" in k:
            assert named[k].grad is None, k
    checked = 0
    for k, gr in c["grads"].items():
        if any(s in k for s in ("classifier.1", "t_pooler", "v_pooler", "c_layer.1.biattention.query1.weight",
                                "imagePredictions.decoder.weight", "v_embeddings.image_embeddings.weight")):
            assert named[k].grad is not None, k
            assert rel(named[k].grad, gr) < 8e-2, k
            checked += 1
    assert checked >= 3


def test_mmbt_registered_model_classification_runs_and_matches_oracle(cpu_models):
    """MMBT classification from the reference's config keys (configs/models/mmbt/classification.yaml + with_features.yaml):
    scores = classifier(dropout(pooled)) on the trunk the MMBT golden already pins; here vs the oracle's restatement."""
    MD = cpu_models
    from oracle import fusion_oracle as O
    cfg = MD.load_model_config("mmbt", overrides={
        "training_head_type": "classification", "num_labels": 2, "direct_features_input": True, "modal_hidden_size": 40,
        "modal_encoder": {"type": "identity", "params": {"in_dim": 40}},
        "text_encoder": {"type": "transformer", "params": {
            "num_segments": 2, "bert_model_name": None, "hidden_size": 64, "num_hidden_layers": 1, "num_attention_heads": 1,
            "intermediate_size": 128, "vocab_size": 50, "max_position_embeddings": 64, "hidden_dropout_prob": 0.0,
            "attention_probs_dropout_prob": 0.0}},
        "losses": [{"type": "cross_entropy"}]})
    assert MD.MMBT.config_path() == "configs/models/mmbt/pretrain.yaml"
    torch.manual_seed(5)
    model = MD.build_model(cfg).eval()
    for p in model.parameters():        # bf16-representable weights: the double computes in bf16 like the kernels
        p.data = p.data.to(torch.bfloat16).float()
    from mmf_b200.sample import SampleList
    g = golden_io.load("mmbt")
    sl = SampleList(input_ids=g["ids"].clone(), input_mask=g["mask"].clone(), segment_ids=g["seg"].clone(),
                    image_feature_0=g["feats"].clone(), targets=torch.tensor([1, 0]), dataset_name="hm", dataset_type="val")
    out = model(sl)
    assert out["scores"].shape == (2, 2) and list(out["losses"]) == ["val/hm/cross_entropy"]
    assert torch.equal(sl["input_ids"], g["shifted_ids"]) and torch.equal(sl["input_mask"], g["shifted_mask"])   # token surgery
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    ocfg = {"num_hidden_layers": 1, "num_attention_heads": 1, "num_segments": 2}
    seq, pooled = O.mmbt_forward(g["feats"], g["ids"], g["mask"], g["seg"],
                                 {k[len("model.bert.mmbt."):]: v for k, v in sd.items() if k.startswith("model.bert.mmbt.")}, ocfg)[:2]
    h = O.gelu_erf(O.linear(pooled, sd, "model.classifier.0.dense"))
    h = O.layer_norm(h, sd, "model.classifier.0.LayerNorm")
    ref = O.linear(h, sd, "model.classifier.1")
    assert rel(out["scores"], ref) < 3e-2


@pytest.fixture()
def reference_configs(tmp_path):
    """the reference's model YAML files (tests/golden/model_configs.json: their parsed documents, written back as YAML)
    under a stand-in mmf root"""
    import json

    import yaml
    with open(os.path.join(GOLD, "model_configs.json")) as fh:
        docs = json.load(fh)
    for relpath, doc in docs.items():
        path = tmp_path / relpath
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text(yaml.safe_dump(doc, sort_keys=False))
    return str(tmp_path)


def test_restated_defaults_equal_the_reference_yaml(cpu_models, reference_configs):
    """MODEL_DEFAULTS is a restatement: pin it to the YAML files it cites, read with the module's own YAML loader"""
    MD = cpu_models
    REF = reference_configs
    import mmf_b200.mmft  # noqa: F401  (adds the mmf_transformer defaults)
    for name, rel_path in (("visual_bert", "configs/models/visual_bert/defaults.yaml"),
                           ("vilbert", "configs/models/vilbert/defaults.yaml"), ("mmbt", "configs/models/mmbt/defaults.yaml"),
                           ("mmf_transformer", "configs/models/mmf_transformer/defaults.yaml")):
        doc = MD.read_yaml_with_includes(os.path.join(REF, rel_path), REF)
        block = MD._resolve_interpolations(doc["model_config"][name], doc)
        assert dict(MD.ConfigNode(MD.MODEL_DEFAULTS[name])) == dict(MD.ConfigNode(block)), name
    # `includes:` + override order: classification.yaml = defaults + training_head_type
    c = MD.load_model_config("visual_bert", yaml_path="configs/models/visual_bert/classification.yaml", mmf_root=REF)
    assert c.training_head_type == "classification" and c.visual_embedding_dim == 2048
    c = MD.load_model_config("mmbt", yaml_path="configs/models/mmbt/classification.yaml", mmf_root=REF)
    assert c.training_head_type == "classification" and c.losses[0]["type"] == "cross_entropy"
    c = MD.load_model_config("mmbt", yaml_path="configs/models/mmbt/with_features.yaml", mmf_root=REF)
    assert c.direct_features_input is True and c.modal_encoder.type == "finetune_faster_rcnn_fpn_fc7"
