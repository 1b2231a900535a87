"""bench.py host logic that needs no GPU: the algorithmic FLOP counts the throughput / roofline figures are built on
(pinned to BASELINE.md's table), the workload registry, and the default launch mode per configuration."""
import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


@pytest.fixture(scope="module")
def bench():
    return importlib.import_module("bench")


@pytest.mark.parametrize("name,gf,tokens", [("visual_bert", 122.9, 228), ("vilbert", 45.7, 72), ("mmbt", None, 122),
                                            ("mmft", None, 324), ("uniter_large", None, 120)])
def test_workload_flops_match_the_baseline_table(bench, name, gf, tokens):
    """fwd+bwd GFLOP per sample = 3 x forward (BASELINE.md, hot-path table); tokens per sample as SURVEY.md 8a lists them"""
    wl = bench.WORKLOADS[name]()
    assert wl.tokens_per_sample() == tokens
    got = 3 * wl.fwd_flops() / 1e9
    assert got > 0
    if gf is not None:
        assert abs(got - gf) / gf < 2e-3, (name, got)


def test_reference_arm_and_multi_gpu_runs_are_eager(bench, monkeypatch):
    """the CUDA-graph launch mode is a single-GPU default for the workloads it was validated with; everything else is eager"""
    import argparse

    def decide(workload, world, profile=False, impl="b200"):
        # the expression of bench.main(), kept in one place there; mirrored here on its inputs
        return (world == 1 and not profile and impl == "b200" and workload in ("visual_bert", "mmbt", "vilbert"))
    assert decide("visual_bert", 1) and decide("mmbt", 1) and decide("vilbert", 1)
    assert not decide("visual_bert", 8) and not decide("mmft", 1) and not decide("visual_bert", 1, profile=True)
    assert not decide("visual_bert", 1, impl="reference")
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'args.workload in ("visual_bert", "mmbt", "vilbert")' in src and 'not args.profile and args.impl == "b200"' in src
    assert isinstance(argparse.ArgumentParser(), argparse.ArgumentParser)


def test_kept_traffic_is_reported_only_for_the_batch_it_was_captured_at(bench):
    tr, src = bench.kept_traffic("visual_bert", 166)
    assert tr is not None and tr > 4e8 and "ncu" in src            # profiles/dominant_traffic.json: 63 MB read + 406 MB written
    assert bench.kept_traffic("visual_bert", 64) == (None, None)
    assert bench.kept_traffic("no_such_workload", 166) == (None, None)


def test_dump_outputs_stays_within_its_budget_and_samples_reproducibly(bench, monkeypatch, tmp_path):
    import numpy as np
    import torch
    monkeypatch.setattr(bench, "DUMP_BYTES", 3 * (128 + 4 * 1000))
    big = torch.randn(40, 50)
    arrays = {"loss": torch.tensor(1.25), "grad.small": torch.arange(6.0).reshape(2, 3), "grad.big": big}
    total = bench.dump_outputs(str(tmp_path / "a"), arrays)
    assert total <= bench.DUMP_BYTES
    loss, small, sample = (np.load(tmp_path / "a" / (n + ".npy")) for n in ("loss", "grad.small", "grad.big"))
    assert loss.dtype == np.float64 and loss.shape == () and float(loss) == 1.25
    assert small.dtype == np.float32 and np.array_equal(small, np.arange(6.0).reshape(2, 3))
    assert sample.dtype == np.float32 and sample.shape == (1000,) and np.isin(sample, big.numpy()).all()
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    assert np.array_equal(np.load(tmp_path / "b" / "grad.big.npy"), sample)
