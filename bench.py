#!/usr/bin/env python
"""Benchmark of the multimodal-fusion block (forward + backward), BASELINE.json metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--workload NAME] [--impl reference] [--dump-outputs DIR]

Default workload (config.workload): BASELINE.json configs[1] - VisualBERT (visual_bert/pretrain) trunk, 12L/768/12h/3072,
128 text tokens + 100 regions x 2048 per sample, bf16 compute, dropout 0.1 (train mode), synthetic SampleList,
random-init weights.  A "step" is one forward+backward of the fusion block (region projection + embeddings +
12 layers; loss = fixed random projection of the sequence output, BASELINE.md 4) over one batch.
Other named configs, one JSON line each, same timing rules (`--workload`):
    mmbt          configs[0]  MMBT 1 layer, 100 regions + 20 tokens, batch 2 (the reference's CPU-runnable case)
    vilbert       configs[2]  ViLBERT 12t + 6v + 6 co-attention layers, 36 regions + 36 tokens
    mmft          configs[3]  MMFTransformer backend 12L/768, 128 tokens + 196 patch embeddings
    uniter_large  configs[4]  UNITER 24L/1024/16h/4096, 100 regions + 20 tokens, batch 256

  value : samples/s with the step's inputs already resident in HBM (CUDA-event timed, max over ranks)
  e2e   : the same through the public module API with HOST (pinned) inputs: H2D of ids/masks/features and a
          D2H read of the loss inside the timed region
  roofline     : dominant kernel (the tcgen05 GEMM at the workload's FFN-up shape) timed alone with CUDA events,
                 algorithmic FLOPs / duration vs MEASURED_PEAKS.json bf16 peak; `traffic` from the kept ncu capture
  roofline_hbm : the largest HBM-bound kernel (fused LayerNorm backward) timed alone, algorithmic bytes / duration vs the
                 measured copy bandwidth
  parity       : before timing, the model in eval mode on a small batch against the CPU arm with the SAME weights
  cpu_baseline : the reference's own implementation (its files, staged under oracle/_ref by oracle/build_ref.py and run
                 through oracle/ref_loader.py: kind "reference"), else the oracle restatement (kind "port"), fp32, all host
                 threads, on a bounded sample
  --impl reference : times that CPU arm alone, same metric / config / JSON shape.
  --dump-outputs DIR : after the device-resident timed steps, writes what the last of them computed - the loss and every
                 parameter gradient - as DIR/<name>.npy (see dump_outputs), so that two builds can be compared output for
                 output: with the same arguments the weights, inputs and dropout masks are the same from run to run.

N > 1 (torchrun): weak scaling, batch per GPU fixed, gradients of every rank averaged with NCCL all-reduce on
slices of the flat gradient buffer overlapped with the backward (mmf_b200.ddp).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

VOCAB = 30522


def layer_flops(S, H, I, Skv=None):
    """forward FLOPs of one BERT-type layer per sample (SURVEY.md 8d): projections + attention + FFN"""
    Skv = S if Skv is None else Skv
    return 8 * S * H * H + 4 * S * Skv * H + 4 * S * H * I


def bert_config(hidden, heads, inter, layers, p, **extra):
    d = dict(hidden_size=hidden, num_attention_heads=heads, intermediate_size=inter, num_hidden_layers=layers,
             vocab_size=VOCAB, max_position_embeddings=512, type_vocab_size=2, hidden_dropout_prob=p,
             attention_probs_dropout_prob=p, layer_norm_eps=1e-12, hidden_act="gelu", initializer_range=0.02, pad_token_id=0)
    d.update(extra)
    return types.SimpleNamespace(**d)


def _ref_available():
    """the reference's files staged under oracle/_ref by build() (oracle/build_ref.py); the CPU arms load them from there"""
    try:
        from oracle import build_ref
        if not build_ref.available():
            return False
        os.environ.setdefault("MMF_REFERENCE_ROOT", build_ref.DST)
        return True
    except Exception:
        return False


class _Attr(dict):
    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)

    def __setattr__(self, k, v):
        self[k] = v


# --------------------------------------------------------------------------------------------------------
# workloads
# --------------------------------------------------------------------------------------------------------
class Workload:
    name = ""
    default_batch = 64
    cpu_batch = 8
    hidden, inter = 768, 3072

    def describe(self):
        raise NotImplementedError

    def fwd_flops(self):
        raise NotImplementedError

    def tokens_per_sample(self):
        raise NotImplementedError

    # product side
    def build(self, p_drop):
        raise NotImplementedError

    def host_batch(self, B, seed):
        raise NotImplementedError

    def aux(self, B, dev, gen_seed=99):
        raise NotImplementedError

    def loss(self, net, batch, aux):
        raise NotImplementedError

    # CPU side: returns (module, call(batch) -> list of output tensors, kind)
    def cpu_model(self, p_drop):
        raise NotImplementedError

    def weights_for_cpu(self, model):
        """state_dict of the product model under the reference module's key names"""
        return model.state_dict()


def _pin(d):
    out = {}
    for k, v in d.items():
        out[k] = _pin(v) if isinstance(v, dict) else v.pin_memory()
    return out


def to_device(d, dev):
    out = {}
    for k, v in d.items():
        out[k] = to_device(v, dev) if isinstance(v, dict) else v.to(dev, non_blocking=True)
    return out


def tensors_of(d):
    for v in d.values():
        if isinstance(v, dict):
            yield from tensors_of(v)
        else:
            yield v


def h2d_bytes(d):
    return sum(t.numel() * t.element_size() for t in tensors_of(d))


class VisualBertWL(Workload):
    name = "visual_bert"
    default_batch = 166
    T, R, FEAT, H, HEADS, I, L = 128, 100, 2048, 768, 12, 3072, 12
    hidden, inter = 768, 3072

    def describe(self):
        return ("VisualBERT visual_bert/pretrain trunk 12L/768/12h/3072, 128 tokens + 100 regions x 2048 "
                "(BASELINE.json configs[1]); fwd+bwd of region projection + embeddings + 12 fusion layers")

    def tokens_per_sample(self):
        return self.T + self.R

    def fwd_flops(self):
        return self.L * layer_flops(self.T + self.R, self.H, self.I) + 2 * self.R * self.FEAT * self.H

    def config(self, p):
        return bert_config(self.H, self.HEADS, self.I, self.L, p, visual_embedding_dim=self.FEAT)

    def build(self, p):
        from mmf_b200.visual_bert import B200VisualBERT
        return B200VisualBERT(self.config(p))

    def host_batch(self, B, seed):
        import torch
        g = torch.Generator().manual_seed(seed)
        T, R = self.T, self.R
        ids = torch.randint(0, VOCAB, (B, T), generator=g)
        lens = torch.randint(T // 2, T + 1, (B,), generator=g)
        mask = (torch.arange(T)[None, :] < lens[:, None]).long()
        feats = torch.randn(B, R, self.FEAT, generator=g).abs()
        maxf = torch.randint(R // 2, R + 1, (B,), generator=g)
        return {"input_ids": ids, "input_mask": mask, "segment_ids": torch.zeros(B, T, dtype=torch.long),
                "image_feature_0": feats, "image_info_0": {"max_features": maxf}}

    def aux(self, B, dev, gen_seed=99):
        import torch
        g = torch.Generator().manual_seed(gen_seed)
        return [torch.randn(B, self.T + self.R, self.H, generator=g).to(dev)]

    def loss(self, net, batch, aux):
        return (net(batch)["sequence_output"] * aux[0]).sum()

    def cpu_model(self, p):
        import torch
        if _ref_available():
            from oracle import ref_loader as R
            from transformers import BertConfig
            vb = R.visual_bert()
            orig = vb.VisualBERTBase.init_weights
            vb.VisualBERTBase.init_weights = lambda self: None          # see ref_loader.visual_bert()
            try:
                cfg = BertConfig(hidden_size=self.H, num_attention_heads=self.HEADS, intermediate_size=self.I,
                                 num_hidden_layers=self.L, vocab_size=VOCAB, max_position_embeddings=512,
                                 hidden_dropout_prob=p, attention_probs_dropout_prob=p)
                m = vb.VisualBERTBase(cfg, visual_embedding_dim=self.FEAT)
            finally:
                vb.VisualBERTBase.init_weights = orig
            _init_ref(m)

            def call(b):
                R_ = b["image_feature_0"].shape[1]
                image_mask = (torch.arange(R_).expand(b["image_feature_0"].shape[:-1]) <
                              b["image_info_0"]["max_features"].unsqueeze(-1)).long()        # visual_bert.py:538-556
                att = torch.cat((b["input_mask"], image_mask), dim=-1)
                seq, _, _ = m(b["input_ids"], att, b["segment_ids"], b["image_feature_0"], torch.zeros_like(image_mask))
                return [seq]
            return m, call, "reference"
        # oracle restatement (kind "port")
        from oracle import fusion_oracle as O
        sd = O.make_encoder_weights(self.L, self.H, self.I, seed=0, prefix="encoder.layer")
        g = torch.Generator().manual_seed(1)
        sd["emb.word_embeddings.weight"] = torch.randn(VOCAB, self.H, generator=g) * 0.02
        sd["emb.position_embeddings.weight"] = torch.randn(512, self.H, generator=g) * 0.02
        sd["emb.token_type_embeddings.weight"] = torch.randn(2, self.H, generator=g) * 0.02
        sd["emb.token_type_embeddings_visual.weight"] = torch.randn(2, self.H, generator=g) * 0.02
        sd["emb.position_embeddings_visual.weight"] = torch.randn(512, self.H, generator=g) * 0.02
        sd["emb.projection.weight"] = torch.randn(self.H, self.FEAT, generator=g) * 0.02
        sd["emb.projection.bias"] = torch.zeros(self.H)
        sd["emb.LayerNorm.weight"] = torch.ones(self.H)
        sd["emb.LayerNorm.bias"] = torch.zeros(self.H)
        holder = torch.nn.ParameterDict({k.replace(".", "__"): torch.nn.Parameter(v) for k, v in sd.items()})
        live = {k: holder[k.replace(".", "__")] for k in sd}

        def call(b):
            _, vtype, att = O.visual_bert_masks(b["input_mask"], b["image_info_0"]["max_features"], self.R)
            keep, masks = None, None
            if p > 0 and holder.training:
                keep = "rng"
                masks = [{"attn": "rng", "self_out": "rng", "out": "rng"} for _ in range(self.L)]
            emb = O.visio_linguistic_embeddings(b["input_ids"], b["segment_ids"], b["image_feature_0"], vtype, live, "emb",
                                                keep=keep, p=p)
            return [O.bert_encoder(emb, O.extended_attention_mask(att), live, "encoder", self.L, self.HEADS, masks, p, p)]
        return holder, call, "port"

    def weights_for_cpu(self, model):
        return model.bert.state_dict()


class VilbertWL(Workload):
    name = "vilbert"
    default_batch = 512
    cpu_batch = 16
    T, R, FEAT = 36, 36, 2048
    hidden, inter = 768, 3072

    def describe(self):
        return ("ViLBERT two-stream co-attention: text 12L/768/12h/3072, image 6L/1024/8h/1024, 6 connection layers "
                "1024/8h (d=128), 36 regions x 2048 (+5 location features) + 36 tokens (BASELINE.json configs[2])")

    def tokens_per_sample(self):
        return self.T + self.R

    def fwd_flops(self):
        T, R = self.T, self.R
        t = 12 * layer_flops(T, 768, 3072)
        v = 6 * layer_flops(R, 1024, 1024)
        bi = 2 * T * 768 * 1024 * 3 + 2 * R * 1024 * 1024 * 3 + 2 * (4 * T * R * 1024) + 2 * T * 1024 * 768 \
            + 2 * R * 1024 * 1024 + 4 * T * 768 * 3072 + 4 * R * 1024 * 1024
        return t + v + 6 * bi + 2 * R * self.FEAT * 1024 + 2 * R * 5 * 1024

    def config(self, p):
        # mmf/configs/models/vilbert/defaults.yaml:11-49
        return bert_config(768, 12, 3072, 12, p, v_feature_size=self.FEAT, v_target_size=1601, v_hidden_size=1024,
                           v_num_hidden_layers=6, v_num_attention_heads=8, v_intermediate_size=1024, bi_hidden_size=1024,
                           bi_num_attention_heads=8, bi_intermediate_size=1024, v_attention_probs_dropout_prob=p,
                           v_hidden_dropout_prob=p, v_biattention_id=[0, 1, 2, 3, 4, 5], t_biattention_id=[6, 7, 8, 9, 10, 11],
                           v_hidden_act="gelu", fast_mode=False, with_coattention=True, dynamic_attention=False,
                           fixed_t_layer=0, fixed_v_layer=0, in_batch_pairs=False, bi_attention_type=1,
                           v_initializer_range=0.02, fusion_method="mul", pooling_method="mul", task_specific_tokens=False,
                           visualization=False, visual_target=0, objective=0, num_negative=128, model="bert")

    def build(self, p):
        from mmf_b200.vilbert import B200ViLBERTBase
        return B200ViLBERTBase(self.config(p))

    def host_batch(self, B, seed):
        import torch
        g = torch.Generator().manual_seed(seed)
        T, R = self.T, self.R
        ids = torch.randint(0, VOCAB, (B, T), generator=g)
        lens = torch.randint(T // 2, T + 1, (B,), generator=g)
        tmask = (torch.arange(T)[None, :] < lens[:, None]).long()
        feats = torch.randn(B, R, self.FEAT, generator=g).abs()
        loc = torch.rand(B, R, 5, generator=g)
        nreg = torch.randint(R // 2, R + 1, (B,), generator=g)
        return {"input_ids": ids, "input_mask": tmask, "image_feature_0": feats, "bbox": loc, "max_features": nreg}

    def aux(self, B, dev, gen_seed=99):
        import torch
        g = torch.Generator().manual_seed(gen_seed)
        return [torch.randn(B, self.T, 768, generator=g).to(dev), torch.randn(B, self.R, 1024, generator=g).to(dev)]

    @staticmethod
    def _image_mask(b):
        import torch
        f = b["image_feature_0"]
        return (torch.arange(f.size(-2), device=f.device).expand(*f.size()[:-1]) < b["max_features"].unsqueeze(-1)).long()

    def loss(self, net, batch, aux):
        t_out, v_out, _ = net(batch["input_ids"], batch["image_feature_0"], batch["bbox"],
                              attention_mask=batch["input_mask"], image_attention_mask=self._image_mask(batch))
        return (t_out * aux[0]).sum() + (v_out * aux[1]).sum()

    def cpu_model(self, p):
        if not _ref_available():
            return None, None, None
        from oracle import ref_loader as R
        from transformers import BertConfig
        vil = R.vilbert()
        orig = vil.ViLBERTBase.init_weights
        vil.ViLBERTBase.init_weights = lambda self: None
        try:
            c = vars(self.config(p))
            cfg = BertConfig(**{k: v for k, v in c.items()})
            m = vil.ViLBERTBase(cfg)
        finally:
            vil.ViLBERTBase.init_weights = orig
        _init_ref(m)

        def call(b):
            out = m(b["input_ids"], b["image_feature_0"], b["bbox"], None, b["input_mask"], self._image_mask(b))
            return [out[0], out[1]]
        return m, call, "reference"


class MmbtWL(Workload):
    name = "mmbt"
    default_batch = 2
    cpu_batch = 2
    T, R, FEAT, H, I, L = 20, 100, 2048, 768, 3072, 1

    def describe(self):
        return ("MMBT hateful_memes-style trunk, 1 layer/768/12h/3072, [CLS] + 100 regions x 2048 + [SEP] + 20 tokens = 122 "
                "positions (BASELINE.json configs[0]); fwd+bwd of modal projection + embeddings + encoder")

    def tokens_per_sample(self):
        return self.T + self.R + 2

    def fwd_flops(self):
        return self.L * layer_flops(self.T + self.R + 2, self.H, self.I) + 2 * self.R * self.FEAT * self.H

    def config(self, p):
        return bert_config(self.H, 12, self.I, self.L, p, modal_hidden_size=self.FEAT)

    def build(self, p):
        from mmf_b200.mmbt import B200MMBTBase
        return B200MMBTBase(self.config(p))

    def host_batch(self, B, seed):
        import torch
        g = torch.Generator().manual_seed(seed)
        T = self.T
        ids = torch.randint(1000, VOCAB, (B, T), generator=g)
        ids[:, 0] = 101
        lens = torch.randint(T // 2, T + 1, (B,), generator=g)
        mask = (torch.arange(T)[None, :] < lens[:, None]).long()
        ids[torch.arange(B), lens - 1] = 102
        return {"input_ids": ids, "input_mask": mask, "segment_ids": torch.zeros(B, T, dtype=torch.long),
                "image_feature_0": torch.randn(B, self.R, self.FEAT, generator=g).abs()}

    def aux(self, B, dev, gen_seed=99):
        import torch
        g = torch.Generator().manual_seed(gen_seed)
        return [torch.randn(B, self.T + self.R + 2, self.H, generator=g).to(dev)]

    def loss(self, net, batch, aux):
        return (net(dict(batch))[0] * aux[0]).sum()        # token surgery rewrites input_ids / input_mask: shallow copy

    def cpu_model(self, p):
        if not _ref_available():
            return None, None, None
        import torch
        from oracle import ref_loader as R
        from transformers import BertConfig
        hl, mm = R.hf_layers(), R.mmbt()
        hl.replace_with_jit = lambda: None
        cfg = BertConfig(hidden_size=self.H, num_attention_heads=12, intermediate_size=self.I, num_hidden_layers=self.L,
                         vocab_size=VOCAB, max_position_embeddings=512, hidden_dropout_prob=p, attention_probs_dropout_prob=p)
        cfg.modal_hidden_size = self.FEAT
        m = mm.MMBTModel(cfg, hl.BertModelJit(cfg), torch.nn.Identity())
        _init_ref(m)

        def call(b):
            sl = {"input_ids": b["input_ids"].clone(), "input_mask": b["input_mask"].clone(), "segment_ids": b["segment_ids"]}
            start = sl["input_ids"][:, 0].clone()
            end = mm.MMBTBase.extract_modal_end_token(None, sl)
            tt = torch.full((start.shape[0], 1), 1, dtype=torch.long)
            out = m(b["image_feature_0"], input_ids=sl["input_ids"], modal_start_tokens=start, modal_end_tokens=end,
                    attention_mask=sl["input_mask"], token_type_ids=sl["segment_ids"], modal_token_type_ids=tt)
            return [out[0]]
        return m, call, "reference"

    def weights_for_cpu(self, model):
        return model.mmbt.state_dict()


class MmftWL(Workload):
    name = "mmft"
    default_batch = 116
    T, P, EMB, H, I, L = 128, 196, 768, 768, 3072, 12

    def describe(self):
        return ("MMFTransformer backend 12L/768/12h/3072, 128 text tokens + 196 image patch embeddings x 768 = 324 positions "
                "(BASELINE.json configs[3]; synthetic composition, SURVEY.md 8d: image modality fed pre-computed patch "
                "embeddings with encoder: identity)")

    def tokens_per_sample(self):
        return self.T + self.P

    def fwd_flops(self):
        return self.L * layer_flops(self.T + self.P, self.H, self.I) + 2 * self.P * self.EMB * self.H

    def build(self, p):
        from mmf_b200.mmft_backend import B200TransformerBackend
        cfg = _Attr(modalities=[_Attr(type="text", key="text", position_dim=512, embedding_dim=768, segment_id=0,
                                      layer_norm_eps=1e-12, hidden_dropout_prob=p),
                                _Attr(type="image", key="image", position_dim=196, embedding_dim=self.EMB, segment_id=1,
                                      layer_norm_eps=1e-12, hidden_dropout_prob=p)],
                    token_noise_mean=0.0, token_noise_std=0.01, transformer_config=bert_config(self.H, 12, self.I, self.L, p))
        return B200TransformerBackend(cfg)

    def host_batch(self, B, seed):
        import torch
        g = torch.Generator().manual_seed(seed)
        T = self.T
        lens = torch.randint(T // 2, T + 1, (B,), generator=g)
        return {"text": torch.randint(1, VOCAB, (B, T), generator=g),
                "text_mask": (torch.arange(T)[None, :] < lens[:, None]).long(),
                "image": torch.randn(B, self.P, self.EMB, generator=g)}

    def aux(self, B, dev, gen_seed=99):
        import torch
        g = torch.Generator().manual_seed(gen_seed)
        return [torch.randn(B, self.T + self.P, self.H, generator=g).to(dev)]

    def loss(self, net, batch, aux):
        import torch
        B, dev = batch["text"].shape[0], batch["text"].device
        pos = {"text": torch.arange(self.T, device=dev).unsqueeze(0).expand(B, self.T),
               "image": torch.arange(self.P, device=dev).unsqueeze(0).expand(B, self.P)}
        seg = {"text": torch.zeros(B, self.T, dtype=torch.long, device=dev),
               "image": torch.ones(B, self.P, dtype=torch.long, device=dev)}
        masks = [batch["text_mask"], torch.ones(B, self.P, dtype=torch.long, device=dev)]
        seq, _ = net({"text": batch["text"], "image": batch["image"]}, pos, seg, masks)
        return (seq * aux[0]).sum()

    def cpu_model(self, p):
        return None, None, None


class UniterLargeWL(Workload):
    name = "uniter_large"
    default_batch = 256
    cpu_batch = 4
    T, R, FEAT, H, HEADS, I, L = 20, 100, 2048, 1024, 16, 4096, 24
    hidden, inter = 1024, 4096

    def describe(self):
        return ("UNITER-large trunk 24L/1024/16h/4096, 100 regions x 2048 (+7 box features) + 20 tokens "
                "(BASELINE.json configs[4])")

    def tokens_per_sample(self):
        return self.T + self.R

    def fwd_flops(self):
        return self.L * layer_flops(self.T + self.R, self.H, self.I) + 2 * self.R * self.FEAT * self.H

    def build(self, p):
        from mmf_b200.uniter import B200UNITERModelBase
        return B200UNITERModelBase(bert_config(self.H, self.HEADS, self.I, self.L, p), img_dim=self.FEAT, hidden_dropout_prob=p)

    def host_batch(self, B, seed):
        import torch
        g = torch.Generator().manual_seed(seed)
        T, R = self.T, self.R
        lens = torch.randint(T // 2, T + 1, (B,), generator=g)
        nreg = torch.randint(R // 2, R + 1, (B,), generator=g)
        att = torch.cat([(torch.arange(T)[None, :] < lens[:, None]).long(), (torch.arange(R)[None, :] < nreg[:, None]).long()], 1)
        return {"input_ids": torch.randint(1, VOCAB, (B, T), generator=g), "img_feat": torch.randn(B, R, self.FEAT, generator=g).abs(),
                "img_pos_feat": torch.rand(B, R, 7, generator=g), "attention_mask": att}

    def aux(self, B, dev, gen_seed=99):
        import torch
        g = torch.Generator().manual_seed(gen_seed)
        return [torch.randn(B, self.T + self.R, self.H, generator=g).to(dev)]

    def loss(self, net, batch, aux):
        import torch
        pos_ids = torch.arange(self.T, device=batch["input_ids"].device).unsqueeze(0)       # [1, T] like uniter.py:732-737
        out = net(batch["input_ids"], pos_ids, batch["img_feat"], batch["img_pos_feat"], batch["attention_mask"])
        return (out.final_layer * aux[0]).sum()

    def cpu_model(self, p):
        if not _ref_available():
            return None, None, None
        import torch
        from oracle import ref_loader as R
        from transformers import BertConfig
        from transformers.models.bert.modeling_bert import BertEmbeddings, BertPooler
        un, hl = R.uniter(), R.hf_layers()
        cfg = BertConfig(hidden_size=self.H, num_attention_heads=self.HEADS, intermediate_size=self.I, num_hidden_layers=self.L,
                         vocab_size=VOCAB, max_position_embeddings=512, hidden_dropout_prob=p, attention_probs_dropout_prob=p)
        m = un.UNITERModelBase.__new__(un.UNITERModelBase)
        torch.nn.Module.__init__(m)
        m.text_embeddings = BertEmbeddings(cfg)
        m.img_embeddings = un.UNITERImageEmbeddings(img_dim=self.FEAT, hidden_size=self.H, hidden_dropout_prob=p)
        m.encoder = hl.BertEncoderJit(cfg)
        m.pooler = BertPooler(cfg)
        _init_ref(m)

        def call(b):
            pos_ids = torch.arange(self.T).unsqueeze(0)
            return [m(b["input_ids"], pos_ids, b["img_feat"], b["img_pos_feat"], b["attention_mask"]).final_layer]
        return m, call, "reference"


WORKLOADS = {w.name: w for w in (VisualBertWL, VilbertWL, MmbtWL, MmftWL, UniterLargeWL)}


def _init_ref(m):
    """reference init: normal(0, 0.02) weights, zero biases, LayerNorm (1, 0) - transformers/base.py:213-223"""
    import torch
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, (torch.nn.Linear, torch.nn.Embedding)):
                mod.weight.copy_(torch.randn(mod.weight.shape, generator=g) * 0.02)
                if isinstance(mod, torch.nn.Linear) and mod.bias is not None:
                    mod.bias.zero_()
            elif isinstance(mod, torch.nn.LayerNorm):
                mod.weight.fill_(1.0)
                mod.bias.zero_()


class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md)"""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


def usable_cores():
    """host threads this process may actually use: affinity mask capped by the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


# --------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own files (oracle/_ref through oracle/ref_loader.py), else the oracle restatement
# --------------------------------------------------------------------------------------------------------
def run_cpu_arm(wl, steps, warmup, B, p_drop):
    """-> (samples/s, ms/step, threads, kind, sample description) or None when no CPU implementation is at hand"""
    import torch
    cores = usable_cores()
    torch.set_num_threads(cores)
    m, call, kind = wl.cpu_model(p_drop)
    if m is None:
        return None
    m.train()
    batch = wl.host_batch(B, 1234)
    aux = wl.aux(B, "cpu")

    def step():
        for p_ in m.parameters():
            p_.grad = None
        outs = call(batch)
        loss = sum((o * a).sum() for o, a in zip(outs, aux))
        loss.backward()
        return float(loss.detach())
    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    what = "the reference's own files (oracle/_ref via oracle/ref_loader.py)" if kind == "reference" else "oracle/fusion_oracle.py"
    return B / med, med * 1e3, torch.get_num_threads(), kind, "%d timed steps of batch %d of the same workload, fp32, %s" % (
        steps, B, what)


def parity_check(wl, model, dev, B=4):
    """eval-mode forward of the product on a small batch vs the CPU arm carrying the SAME weights (relative L2)"""
    import torch
    try:
        m, call, kind = wl.cpu_model(0.0)
        if m is None:
            return {"checked": False, "why": "no CPU implementation for this workload on this box"}
        res = m.load_state_dict({k: v.detach().float().cpu() for k, v in wl.weights_for_cpu(model).items()}, strict=False) \
            if kind == "reference" else None
        if kind != "reference":
            return {"checked": False, "why": "reference files not staged (oracle/_ref); the port arm keeps its own weights"}
        missing = [k for k in res.missing_keys if not k.endswith("position_ids")]
        m.eval()
        model.eval()
        batch = wl.host_batch(B, 4321)
        with torch.no_grad():
            ref = call(batch)
            got = _forward_outputs(wl, model, to_device(batch, dev))
        model.train()
        errs = [float(((g.float().cpu() - r).norm() / r.norm()).item()) for g, r in zip(got, ref)]
        # 12+ post-LN layers in bf16 against the fp32 reference: the reference's own bf16-vs-fp32 drift at this depth is
        # 1.25e-2 (SURVEY.md 8d), so the end-to-end bar is 2.5e-2; per-layer parity (1e-2) is what tests/ assert
        return {"checked": True, "against": kind, "batch": B, "rel_l2": errs, "bar": 2.5e-2, "ok": max(errs) < 2.5e-2,
                "missing_keys": len(missing), "unexpected_keys": len(res.unexpected_keys)}
    except Exception as e:      # the bench must still produce its line
        return {"checked": False, "why": "parity check raised %s: %s" % (type(e).__name__, str(e)[:200])}


def _forward_outputs(wl, model, batch):
    """the product's outputs for `batch` (list of tensors, same order as the CPU arm's)"""
    if wl.name == "visual_bert":
        return [model(batch)["sequence_output"]]
    if wl.name == "vilbert":
        t, v, _ = model(batch["input_ids"], batch["image_feature_0"], batch["bbox"], attention_mask=batch["input_mask"],
                        image_attention_mask=wl._image_mask(batch))
        return [t, v]
    if wl.name == "mmbt":
        return [model(dict(batch))[0]]
    if wl.name == "uniter_large":
        import torch
        pos_ids = torch.arange(wl.T, device=batch["input_ids"].device).unsqueeze(0)
        return [model(batch["input_ids"], pos_ids, batch["img_feat"], batch["img_pos_feat"], batch["attention_mask"]).final_layer]
    raise RuntimeError("no output hook for %s" % wl.name)


def kept_traffic(wl_name, B):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the kept `ncu --set full` capture
    (profiles/dominant_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep): only for the batch it was taken at"""
    path = os.path.join(ROOT, "profiles", "dominant_traffic.json")
    try:
        with open(path) as fh:
            d = json.load(fh)
        e = d.get(wl_name)
        if e and int(e.get("batch", -1)) == int(B):
            return float(e["dram_bytes_read"]) + float(e["dram_bytes_write"]), e.get("source")
    except Exception:
        pass
    return None, None


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes {name: tensor} as <out_dir>/<name>.npy, float32 (a 0-d tensor, the loss, as float64), DUMP_BYTES at most in
    all.  Each array gets an equal share; one with more elements than its share holds is written as a fixed sample of
    them instead (flattened, indices drawn with a generator seeded the same for every array), so two runs or two builds
    store the same positions."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = (DUMP_BYTES // len(arrays) - 128) // 4         # 128: the .npy header
    total = 0
    for name, t in arrays.items():
        t = t.detach()
        if t.dim() == 0:
            a = np.asarray(t.double().cpu().numpy())
        else:
            if t.numel() > cap:
                idx = torch.randint(0, t.numel(), (cap,), generator=torch.Generator().manual_seed(0)).to(t.device)
                t = t.reshape(-1)[idx]
            a = t.float().cpu().numpy()
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a)
        total += os.path.getsize(path)
    assert total <= DUMP_BYTES, total
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default=os.environ.get("MMFB_BENCH_WORKLOAD", "visual_bert"), choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=int(os.environ.get("MMFB_BENCH_BATCH", "0")), help="samples per GPU")
    ap.add_argument("--dropout", type=float, default=0.1)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-batch", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--ddp-mode", default=os.environ.get("MMFB_DDP_MODE", "end"), choices=["end", "bucket"],
                    help="gradient exchange: one all-reduce per flat buffer after the backward, or bucket slices "
                         "overlapped with it (mmf_b200/ddp.py)")
    ap.add_argument("--ddp-payload", default=os.environ.get("MMFB_DDP_PAYLOAD", "fp32"), choices=["fp32", "bf16"],
                    help="dtype of the gradients on the wire (bf16: half the bytes, 2^-9 rounding of the averaged gradients)")
    ap.add_argument("--optimizer", action="store_true",
                    help="also time the step WITH the fused AdamW update (mmf_b200.optim.B200AdamW, BERT parameter groups); "
                         "reported as `with_optimizer`, the headline value stays forward + backward (BASELINE.json metric)")
    ap.add_argument("--graph", dest="graph", action="store_true", default=None,
                    help="replay the step (forward + backward) as ONE CUDA graph (mmf_b200.graphs.GraphedStep): the same C-ABI "
                         "launches recorded by stream capture.  Default: on for a single GPU and the workloads it has been "
                         "validated with (visual_bert, mmbt, vilbert) - ~430 launches of ~45 us host time each are 19 ms per "
                         "step, which a slow host CPU cannot hide behind a 26 ms step (seen as e2e 5530 against value 6323 on "
                         "one lease); single GPU only")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="launch every kernel of the step eagerly")
    ap.add_argument("--profile", action="store_true", help="device-resident steps only (for ncu launch lists)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and the parameter gradients of the last timed step as DIR/<name>.npy (b200 arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 arm computed")

    wl = WORKLOADS[args.workload]()
    if args.graph is None:
        args.graph = (int(os.environ.get("WORLD_SIZE", "1")) == 1 and not args.profile and args.impl == "b200"
                      and args.workload in ("visual_bert", "mmbt", "vilbert"))
    B = args.batch or wl.default_batch
    cpu_B = args.cpu_batch or wl.cpu_batch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    S = wl.tokens_per_sample()
    step_flops = 3 * wl.fwd_flops()
    config = {"workload": wl.describe(), "workload_key": wl.name, "batch_per_gpu": B, "global_batch": B * max(world, 1),
              "seq_len": S, "dropout": args.dropout, "parallelism": "dp%d" % max(world, 1),
              "gflop_per_sample_fwd_bwd": step_flops / 1e9,
              "l2_policy": "activations + weights touched per step exceed the 126 MB L2 at this batch"
                           if B * S >= 8192 else "small batch: the working set fits L2; a 160 MB buffer is zeroed between "
                                                 "timed steps (L2 flush)"}
    if wl.name == "visual_bert":
        config["batch_choice"] = ("166 samples x 228 tokens = 147.8 -> 148 pair tiles of 256 rows: every GEMM of the block is "
                                  "an exact number of waves on 148 SMs (sweep in profiles/README.md)")

    if args.impl == "reference":
        if rank != 0:
            return 0
        cpu_steps = max(1, min(args.steps, 5))
        r = run_cpu_arm(wl, cpu_steps, max(1, min(args.warmup, 1)), cpu_B, args.dropout)
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "no CPU implementation of workload %s on this box" % wl.name}))
            return 0
        v, ms, cores, kind, sample = r
        cfg = dict(config, batch_per_gpu=cpu_B, global_batch=cpu_B, parallelism="cpu x%d threads" % cores,
                   note="bounded sample of the b200 arm's workload: same model / sequence shape, batch %d per step" % cpu_B)
        line = {"impl": "reference", "metric": "multimodal-fusion samples/sec (fwd+bwd)", "value": v, "unit": "samples/s",
                "n_gpus": args.gpus, "steps": cpu_steps, "warmup": 1, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
                "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": kind, "sample": sample},
                "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from mmf_b200 import functional as F, lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)
    model = wl.build(args.dropout).to(dev).train()
    ddp = None
    if world > 1:
        from mmf_b200.ddp import B200DataParallel
        ddp = B200DataParallel(model, mode=args.ddp_mode, payload=args.ddp_payload)
        config["ddp_mode"] = args.ddp_mode
        config["ddp_payload"] = args.ddp_payload
    net = ddp if ddp is not None else model
    host = _pin(wl.host_batch(B, 1234 + rank))
    dev_batch = to_device(host, dev)
    aux = wl.aux(B, dev)
    small = B * S < 8192
    flush = torch.empty(160 << 20, dtype=torch.uint8, device=dev) if small else None

    def step(batch):
        model.zero_grad(set_to_none=True)
        loss = wl.loss(net, batch, aux)
        loss.backward()
        return loss

    if args.graph:
        if world > 1:
            raise SystemExit("--graph is a single-GPU mode")
        from mmf_b200.graphs import GraphedStep
        lc0 = lib.launch_count()
        try:
            graphed = GraphedStep(model, lambda b: wl.loss(net, b, aux), dev_batch, warmup=3)
        except Exception as e:      # the eager step is always available: say what happened and go on
            graphed = None
            args.graph = False
            torch.cuda.synchronize()
            model.zero_grad(set_to_none=True)
            config["step_launch"] = "eager (CUDA graph capture failed: %s)" % (str(e).splitlines()[0][:120] if str(e) else type(e).__name__)
        if graphed is not None:
            graph_launches = (lib.launch_count() - lc0) // 4        # 3 warm-up steps + the captured one: kernels per replay
            config["kernels_per_graph"] = graph_launches
            config["step_launch"] = "one CUDA graph per step (stream capture of the eager step; dropout masks advance through a device counter)"

            def step(batch):        # noqa: F811  (same contract: forward + backward of `batch`, returns the loss)
                return graphed(batch)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    parity = None
    if rank == 0 and not args.no_parity and not args.profile:
        parity = parity_check(wl, model, dev)
    for _ in range(max(3, args.warmup)):
        step(dev_batch)
    barrier()
    # ---------------- device-resident timing ----------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.launch_count()
    barrier()
    if args.profile:
        torch.cuda.profiler.start()    # ncu --profile-from-start off: capture exactly the timed steps
    if small:
        # per-step events so that the L2 flush between steps stays outside the timed intervals
        evs = []
        for _ in range(args.steps):
            flush.zero_()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            last_loss = step(dev_batch)
            b_.record()
            evs.append((a, b_))
        barrier()
        ms_total = sum(a.elapsed_time(b_) for a, b_ in evs)
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            last_loss = step(dev_batch)
        e1.record()
        barrier()
        ms_total = e0.elapsed_time(e1)
    if args.profile:
        torch.cuda.profiler.stop()
    launches = lib.launch_count() - launches0
    if args.graph:
        launches = graph_launches * args.steps      # replays do not pass through the C ABI: kernels recorded at capture x steps
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        outs = {"loss": last_loss}
        outs.update(("grad." + n, p_.grad) for n, p_ in model.named_parameters() if p_.grad is not None)
        dump_outputs(args.dump_outputs, outs)
    if args.profile:
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": ms_total / args.steps, "launches": launches}))
        return 0
    # ---------------- end-to-end timing (host inputs, loss read back) ----------------
    for _ in range(2):
        float(step(to_device(host, dev)).detach())
    barrier()
    # Input pipeline as in the reference trainer (pinned SampleList + non_blocking copies, sample.py:326-370): the H2D of
    # step i+1 is issued on a copy stream while step i computes.  Every step still copies its full inputs H2D and reads
    # its loss back D2H inside the timed region.
    copy_stream = torch.cuda.Stream()

    def prefetch():
        with torch.cuda.stream(copy_stream):
            batch = to_device(host, dev)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return batch, ev

    # Every step's loss is copied D2H into pinned memory and READ on the host; the read of step i happens after step i+1
    # has been enqueued (the trainer's logging does the same), so the host never drains the device queue between steps.
    loss_host = torch.zeros(args.steps, dtype=torch.float32).pin_memory()
    loss_ev = [torch.cuda.Event() for _ in range(args.steps)]
    read_back = []
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    nxt = prefetch()
    for i in range(args.steps):
        batch, ev = nxt
        torch.cuda.current_stream().wait_event(ev)
        if i + 1 < args.steps:
            nxt = prefetch()
        loss = step(batch)
        for t in tensors_of(batch):      # keep the copy-stream allocations alive until the compute stream has used them
            t.record_stream(torch.cuda.current_stream())
        loss_host[i:i + 1].copy_(loss.detach().float().reshape(1), non_blocking=True)      # D2H of the step's result
        loss_ev[i].record()
        if i >= 1:
            loss_ev[i - 1].synchronize()
            read_back.append(float(loss_host[i - 1]))
    loss_ev[args.steps - 1].synchronize()
    read_back.append(float(loss_host[args.steps - 1]))
    f1.record()
    barrier()
    assert len(read_back) == args.steps and all(v == v for v in read_back), "a step's loss was not read back / is NaN"
    ms_e2e = f0.elapsed_time(f1)
    ms_opt = 0.0
    if args.optimizer:
        from mmf_b200.optim import B200AdamW
        decay = [p_ for n_, p_ in model.named_parameters() if not any(k in n_ for k in ("bias", "LayerNorm.weight"))]
        nodecay = [p_ for n_, p_ in model.named_parameters() if any(k in n_ for k in ("bias", "LayerNorm.weight"))]
        opt = B200AdamW([{"params": decay, "weight_decay": 0.01}, {"params": nodecay, "weight_decay": 0.0}], lr=5e-5, eps=1e-6)

        def opt_step(batch):
            loss = wl.loss(net, batch, aux)         # no zero_grad: the gradients alias the flat buffer and are re-zeroed by
            loss.backward()                         # prepare_grads only when .grad was released
            opt.step()
            model.zero_grad(set_to_none=True)
        for _ in range(3):
            opt_step(dev_batch)
        barrier()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record()
        for _ in range(args.steps):
            opt_step(dev_batch)
        o1.record()
        barrier()
        ms_opt = o0.elapsed_time(o1)
    t = torch.tensor([ms_total, ms_e2e, ms_opt], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, ms_opt = t.tolist()
    ms_step = ms_total / args.steps
    value = B * world / (ms_step / 1e3)
    e2e_value = B * world / (ms_e2e / args.steps / 1e3)

    if rank == 0:
        burst, sustained, hbm, how = peaks()
        big = torch.empty(160 << 20, dtype=torch.uint8, device=dev)

        def time_alone(fn, n=13, skip=3):
            ts = []
            for i in range(n):
                big.zero_()   # L2 flush between timed launches
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                fn()
                g1.record()
                torch.cuda.synchronize()
                if i >= skip:
                    ts.append(g0.elapsed_time(g1))
            return statistics.mean(ts)
        # dominant kernel alone: the tcgen05 GEMM at the FFN-up shape [B*S, H] x [I, H]^T (+bias+GELU epilogue)
        M, HID, INTER = B * S, wl.hidden, wl.inter
        a = torch.randn(M, HID, device=dev).to(torch.bfloat16)
        w = (torch.randn(INTER, HID, device=dev) * 0.02).to(torch.bfloat16)
        bias = torch.zeros(INTER, device=dev, dtype=torch.bfloat16)
        o1 = torch.empty(M, INTER, device=dev, dtype=torch.bfloat16)
        o2 = torch.empty_like(o1)
        k_ms = time_alone(lambda: F.gemm(a, w, epi=lib.EPI_BIAS_GELU, bias=bias, out=o1, out2=o2))
        k_flops = 2.0 * M * HID * INTER
        achieved = k_flops / (k_ms * 1e-3) / 1e12
        traffic, traffic_src = kept_traffic(wl.name, B)
        roofline = {"bound": "tensor", "kernel": "gemm_kernel<256,K-major,K-major,BIAS_GELU> FFN-up [%d,%d]x[%d,%d]^T" % (M, HID, INTER, HID),
                    "achieved": achieved, "peak": burst, "unit": "TFLOP/s", "frac": achieved / burst,
                    "peak_source": "%s bf16_tflops (burst: kernel timed alone)" % how,
                    "traffic": traffic, "traffic_source": traffic_src,
                    "kernel_ms": k_ms, "flops_per_launch": k_flops,
                    "step_tflops": step_flops * value / 1e12 / world,
                    "step_frac_of_sustained": step_flops * value / 1e12 / world / sustained}
        # largest HBM-bound kernel alone: LayerNorm backward fused with the dropout backward and the dgamma / dbeta / dbias
        # column sums.  Algorithmic bytes per row: read dx, y (2H each) + keep bits (H/8), write dy, dz (2H each)
        dx = torch.randn(M, HID, device=dev).to(torch.bfloat16)
        y = torch.randn(M, HID, device=dev).to(torch.bfloat16)
        gamma = torch.ones(HID, device=dev, dtype=torch.bfloat16)
        _, mean, rstd = F.layernorm_fwd(y, gamma, torch.zeros_like(gamma))
        bits = F.dropout_bits((M,), HID, 0.1, 1, 0, dev)
        dg, db_, dbias = (torch.zeros(HID, device=dev) for _ in range(3))
        l_ms = time_alone(lambda: F.layernorm_bwd(dx, y, mean, rstd, gamma, dg, db_, dbias=dbias, drop_mask=bits, drop_scale=1 / 0.9))
        l_bytes = M * (8.0 * HID + HID / 8.0 + 8.0)
        roofline_hbm = {"bound": "hbm", "kernel": "layernorm_bwd (+dropout bwd, dgamma/dbeta/dbias) [%d,%d]" % (M, HID),
                        "achieved": l_bytes / (l_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                        "frac": l_bytes / (l_ms * 1e-3) / 1e9 / hbm, "peak_source": "%s hbm_gbs" % how, "traffic": None,
                        "kernel_ms": l_ms, "bytes_per_launch": l_bytes}
        # fused AdamW over a flat fp32 buffer of this model's size: reads p, g, m, v and writes p, m, v (28 B / parameter)
        n_par = (sum(p_.numel() for p_ in model.parameters()) + 7) // 8 * 8
        fp, fg, fm, fv = (torch.zeros(n_par, device=dev) for _ in range(4))
        fg.normal_()
        hp = [{"lr": 5e-5, "weight_decay": 0.01, "step_size": 5e-5, "bc2_sqrt": 1.0}]
        a_ms = time_alone(lambda: F.adamw(fp, fg, fm, fv, hp, beta1=0.9, beta2=0.999, eps=1e-6, mode=0))
        roofline_adamw = {"bound": "hbm", "kernel": "mmfb_adamw over %d parameters (flat fp32 master / grad / m / v)" % n_par,
                          "achieved": 28.0 * n_par / (a_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                          "frac": 28.0 * n_par / (a_ms * 1e-3) / 1e9 / hbm, "kernel_ms": a_ms, "bytes_per_param": 28}
        del a, w, o1, o2, dx, y, big, fp, fg, fm, fv
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            r = run_cpu_arm(wl, 3, 1, cpu_B, args.dropout)
            if r is not None:
                v, ms, cores, kind, sample = r
                cpu = {"value": v, "unit": "samples/s", "cores": cores, "kind": kind, "sample": sample}
        line = {"metric": "multimodal-fusion samples/sec (fwd+bwd)", "value": value, "unit": "samples/s",
                "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": config,
                "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d_bytes(host),
                        "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_hbm": roofline_hbm,
                "roofline_adamw": roofline_adamw, "parity": parity, "cpu_baseline": cpu}
        if args.optimizer:
            line["with_optimizer"] = {"value": B * world / (ms_opt / args.steps / 1e3), "unit": "samples/s",
                                      "ms_per_step": ms_opt / args.steps, "optimizer": "B200AdamW (fused, flat buffers)"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
