"""Registered model plugins on the B200 (through the C ABI): `forward(SampleList) -> scores / losses` of visual_bert and
vilbert against the outputs of the REFERENCE's own registered model classes (tests/golden/models.*.pt), integer tensors with
torch.equal, gradients of the heads and of trunk weights against the reference's autograd."""

import pytest
import torch

from oracle import golden_io

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


def _sample_list(g, dev):
    from mmf_b200.sample import SampleList
    i = g["visual_bert_inputs"]
    return SampleList(input_ids=i["ids"].to(dev), input_mask=i["mask"].to(dev), segment_ids=i["seg"].to(dev),
                      image_feature_0=i["feats"].to(dev), image_info_0={"max_features": i["max_features"].to(dev)},
                      lm_label_ids=i["lm_label_ids"].to(dev), targets=i["targets"].to(dev), dataset_name="golden",
                      dataset_type="train")


@pytest.mark.parametrize("case", ["visual_bert_classification_default", "visual_bert_classification_vqa",
                                  "visual_bert_pretraining_default"])
def test_visual_bert_registered_model(case):
    from mmf_b200 import lib, models as MD
    dev = torch.device("cuda", 0)
    g = golden_io.load("models")
    c = g[case]
    cfg = MD.load_model_config("visual_bert", overrides=dict(c["config"]))
    cfg.losses = [{"type": "cross_entropy"}]
    model = MD.build_model(cfg)
    model.load_state_dict({k: v for k, v in c["state_dict"].items() if k in model.state_dict()})
    model = model.to(dev).eval()
    sl = _sample_list(g, dev)
    n0 = lib.launch_count()
    out = model(sl)
    assert lib.launch_count() > n0
    assert torch.equal(sl["image_mask"].cpu(), c["image_mask"]) and torch.equal(sl["attention_mask"].cpu(), c["attention_mask"])
    if c["scores"] is not None:
        assert rel(out["scores"], c["scores"]) < 1e-2, rel(out["scores"], c["scores"])
        loss = out["losses"]["train/golden/cross_entropy"].sum()
    else:
        assert torch.equal(sl["masked_lm_labels"].cpu(), c["masked_lm_labels"])
        assert rel(out["logits"], c["logits"]) < 1e-2
        loss = out["losses"]["golden/train/masked_lm_loss"]
    assert abs(float(loss.detach()) - float(c["loss"])) < 1e-2 * max(1.0, abs(float(c["loss"])))
    loss.backward()
    named = dict(model.named_parameters())
    worst = 0.0
    for k, gr in c["grads"].items():
        if k in named and named[k].grad is not None and gr.norm() > 1e-6 and gr.dim() == 2:
            worst = max(worst, rel(named[k].grad, gr))
    print("worst 2-D parameter-gradient error", worst)
    assert worst < 3e-2


@pytest.mark.parametrize("head", ["classification", "pretraining"])
def test_vilbert_registered_model(head):
    from mmf_b200 import models as MD
    dev = torch.device("cuda", 0)
    g = golden_io.load("models")
    c = g["vilbert_" + head]
    cfg = MD.load_model_config("vilbert", overrides=dict(c["config"]))
    cfg.losses = [{"type": "cross_entropy"}]
    model = MD.build_model(cfg)
    model.load_state_dict({k: v for k, v in c["state_dict"].items() if k in model.state_dict()})
    model = model.to(dev).eval()
    v = g["vilbert_inputs"]
    sl = _sample_list(g, dev)
    sl["image_labels"] = v["image_labels"].to(dev)
    sl["image_info_0"] = {"max_features": g["visual_bert_inputs"]["max_features"].to(dev), "bbox": v["bbox"].to(dev),
                          "cls_prob": v["cls_prob"].numpy().copy()}
    out = model(sl)
    if head == "classification":
        assert rel(out["scores"], c["scores"]) < 1.5e-2, rel(out["scores"], c["scores"])
        loss = out["losses"]["train/golden/cross_entropy"].sum()
    else:
        for k in c["losses"]:
            assert abs(float(out["losses"][k].detach()) - float(c["losses"][k])) < 1e-2 * max(1.0, abs(float(c["losses"][k]))), k
        loss = sum(x.sum() for x in out["losses"].values())
    loss.backward()
    named = dict(model.named_parameters())
    for k in c["unused"]:
        if "q_dense" in k:
            assert named[k].grad is None, k
    # a classification loss reaches the trunk through ONE pooled token per stream of this 8-token / 5-region fixture: single
    # parameters carry little signal, so the bar is on the whole gradient vector (every 2-D parameter concatenated), with
    # a loose per-parameter ceiling (the 10-token effect documented in tests/test_encoder_gpu.py::check_param_grads)
    num = den = 0.0
    worst, worst_k = 0.0, ""
    for k, gr in c["grads"].items():
        if k in named and named[k].grad is not None and gr.norm() > 1e-6 and gr.dim() == 2 and "word_embeddings" not in k:
            d = (named[k].grad.double().cpu() - gr.double())
            num, den = num + float(d.pow(2).sum()), den + float(gr.double().pow(2).sum())
            e = rel(named[k].grad, gr)
            if e > worst:
                worst, worst_k = e, k
    total = (num / den) ** 0.5
    print("all 2-D parameter gradients: rel %.2e; worst single parameter %.2e (%s)" % (total, worst, worst_k))
    assert total < 3e-2 and worst < 0.25
