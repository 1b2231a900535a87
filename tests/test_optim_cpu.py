"""Optimizer `adam_w` (SURVEY.md 8f item 2, staged): the oracle restatements against the reference's own arithmetic
(tests/golden/adamw.pt, generated from mmf/modules/optimizers.py), and B200AdamW's host logic - parameter groups mapped
onto 8-element blocks of the flat buffers, state views, frozen parameters, parameters outside the packs - over the
kernel test double (tests/fake_kernels.py)."""
import types

import pytest
import torch

from oracle import fusion_oracle as O
from oracle import golden_io

import fake_kernels as FK


def test_oracle_adamw_matches_the_reference_arithmetic_bit_for_bit():
    g = golden_io.load("adamw")
    assert g["adam_w_is"] == "torch.optim.adamw"        # what optimizers.py:8-14 resolves `adam_w` to in this image
    for mode, fn in (("transformers", O.adamw_step_transformers), ("torch", O.adamw_step_torch)):
        ps = [t.clone() for t in g["init"]]
        ms, vs = [torch.zeros_like(t) for t in ps], [torch.zeros_like(t) for t in ps]
        for step, gs in enumerate(g["grads"], 1):
            for p, gr, m, v, wd in zip(ps, gs, ms, vs, g["weight_decay"]):
                fn(p, gr, m, v, step, g["hp"]["lr"], *g["hp"]["betas"], g["hp"]["eps"], wd)
            for p, q in zip(ps, g[mode][step - 1]):
                assert torch.equal(p, q), (mode, step)


@pytest.fixture()
def cpu_engine(monkeypatch):
    import mmf_b200.engine as E
    import mmf_b200.modules as M
    import mmf_b200.optim as OPT
    monkeypatch.setattr(E, "F", FK)
    monkeypatch.setattr(OPT, "F", FK)
    monkeypatch.setattr(M, "_require_cuda", lambda t, what: None)
    yield types.SimpleNamespace(E=E, M=M, OPT=OPT)


def _bert_groups(module, weight_decay=0.01):
    # mmf/utils/modeling.py:18-46
    no_decay = ["bias", "LayerNorm.bias", "LayerNorm.weight"]
    named = list(module.named_parameters())
    return [{"params": [p for n, p in named if not any(nd in n for nd in no_decay)], "weight_decay": weight_decay},
            {"params": [p for n, p in named if any(nd in n for nd in no_decay)], "weight_decay": 0.0}]


class _Model(torch.nn.Module):
    """an engine encoder (parameters in a pack) plus a head outside the pack, one of whose tensors has numel % 8 != 0"""

    def __init__(self, M):
        super().__init__()
        cfg = types.SimpleNamespace(hidden_size=64, num_attention_heads=1, intermediate_size=128, num_hidden_layers=2,
                                    hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, layer_norm_eps=1e-12)
        self.encoder = M.B200BertEncoder(cfg)
        self.head = torch.nn.Linear(64, 3)

    def forward(self, x):
        return self.head(self.encoder(x, None)[0])


@pytest.mark.parametrize("arith", ["transformers", "torch"])
def test_b200_adamw_on_packs_and_loose_parameters_matches_the_oracle(cpu_engine, arith):
    torch.manual_seed(0)
    model = _Model(cpu_engine.M).eval()
    hp = dict(lr=3e-3, betas=(0.9, 0.98), eps=1e-6)
    opt = cpu_engine.OPT.B200AdamW(_bert_groups(model), arithmetic=arith, **hp)
    # reference: the oracle step applied per tensor to detached copies
    ref = {n: p.detach().clone() for n, p in model.named_parameters()}
    rm = {n: torch.zeros_like(p) for n, p in ref.items()}
    rv = {n: torch.zeros_like(p) for n, p in ref.items()}
    wd = {n: (0.0 if any(nd in n for nd in ("bias", "LayerNorm.bias", "LayerNorm.weight")) else 0.01) for n in ref}
    fn = O.adamw_step_transformers if arith == "transformers" else O.adamw_step_torch
    g = torch.Generator().manual_seed(1)
    for step in range(1, 4):
        x = torch.randn(2, 5, 64, generator=g)
        w = torch.randn(2, 5, 3, generator=g)
        model.zero_grad(set_to_none=True)
        (model(x) * w).sum().backward()
        grads = {n: p.grad.detach().clone() for n, p in model.named_parameters()}
        opt.step()
        for n in ref:
            fn(ref[n], grads[n], rm[n], rv[n], step, hp["lr"], *hp["betas"], hp["eps"], wd[n])
        for n, p in model.named_parameters():
            err = (p.detach() - ref[n]).abs().max() / ref[n].abs().max().clamp_min(1e-6)
            assert err < 2e-6, (n, step, float(err))
    pack = model.encoder._runner.pack
    ent = opt._flat[id(pack)]
    qw = model.encoder.layer[0].attention.self.query.weight
    st = opt.state[qw]
    assert st["step"] == 3 and st["exp_avg"].data_ptr() == ent["m"].data_ptr() + 4 * pack.offsets[0]     # views of flat state
    assert opt.state[model.head.bias]["exp_avg"].shape == (3,)                       # numel 3: the torch-op path
    # state_dict round trip keeps torch's layout and is re-adopted into fresh flat buffers
    sd = opt.state_dict()
    opt2 = cpu_engine.OPT.B200AdamW(_bert_groups(model), arithmetic=arith, **hp)
    opt2.load_state_dict(sd)
    model.zero_grad(set_to_none=True)
    x = torch.randn(2, 5, 64, generator=g)
    (model(x) * torch.randn(2, 5, 3, generator=g)).sum().backward()
    before = qw.detach().clone()
    grad = qw.grad.detach().clone()
    m3, v3 = rm["encoder.layer.0.attention.self.query.weight"].clone(), rv["encoder.layer.0.attention.self.query.weight"].clone()
    opt2.step()
    fn(before, grad, m3, v3, 4, hp["lr"], *hp["betas"], hp["eps"], 0.01)
    assert (qw.detach() - before).abs().max() < 2e-6 * before.abs().max()


def test_b200_adamw_leaves_parameters_it_was_not_given_untouched(cpu_engine):
    torch.manual_seed(2)
    model = _Model(cpu_engine.M).eval()
    frozen = [p for n, p in model.encoder.named_parameters() if n.startswith("layer.0.")]
    trained = [p for n, p in model.encoder.named_parameters() if n.startswith("layer.1.")]
    opt = cpu_engine.OPT.B200AdamW(trained, lr=1e-2, arithmetic="transformers")
    (model(torch.randn(2, 5, 64)) ** 2).sum().backward()
    f0 = [p.detach().clone() for p in frozen]
    t0 = [p.detach().clone() for p in trained]
    opt.step()
    assert all(torch.equal(a, p.detach()) for a, p in zip(f0, frozen))
    assert all(not torch.equal(a, p.detach()) for a, p in zip(t0, trained))
    with pytest.raises(ValueError):
        cpu_engine.OPT.B200AdamW(trained, lr=-1.0)
