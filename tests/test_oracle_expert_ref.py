"""Pin oracle.moe_oracle.expert_ffn (D1-D3, SURVEY §8a) against the reference's OWN expert modules.

  * test_oracle_matches_reference_golden: always runs; tests/golden/expert_ffn_ref.pt was produced by
    /root/reference/core/parallel/expert_module.cpp compiled as-is (tests/golden/make_expert_golden.py).
  * test_oracle_matches_live_reference_module: the same module on seeded random shapes of every expert type and dtype;
    tests/golden/expert_ffn_live_ref.pt holds its outputs (tests/golden/make_reference_golden.py).
Bit equality is demanded: both sides call the same ATen operators on the CPU.
"""
from __future__ import annotations

import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))

import expert_cases as C  # noqa: E402
from oracle import moe_oracle as O  # noqa: E402
from reference_cases import SHAPES, rand_case, seed_of  # noqa: E402

GOLD = torch.load(os.path.join(HERE, "golden", "expert_ffn_ref.pt"))
LIVE = torch.load(os.path.join(HERE, "golden", "expert_ffn_live_ref.pt"))


@pytest.mark.parametrize("name", sorted(C.CASES))
def test_oracle_matches_reference_golden(name):
    torch.set_num_threads(1)
    et, di, ws, x = C.make_case(name)
    g = GOLD[name]
    assert abs(sum(float(w.double().abs().sum()) for w in ws) - g["wsum"]) < 1e-9, "weight generator drifted"
    assert torch.equal(x, g["x"])
    y = O.expert_ffn(x, ws, et)
    assert y.dtype == g["y"].dtype and y.shape == g["y"].shape
    assert torch.equal(y, g["y"]), f"{name}: max |diff| {(y.float() - g['y'].float()).abs().max()}"


@pytest.mark.parametrize("et", [0, 1, 2, 3, 4, 5])
@pytest.mark.parametrize("di", [0, 1, 2])
def test_oracle_matches_live_reference_module(et, di):
    torch.set_num_threads(1)
    dt = C.DT[di]
    assert len(LIVE[(et, di)]) == len(SHAPES)
    for i, (H, I, n) in enumerate(SHAPES):
        ws, x = rand_case(et, dt, H, I, n, seed_of(et, di, i))
        y_ref = LIVE[(et, di)][i]
        y = O.expert_ffn(x, ws, et)
        assert y.dtype == y_ref.dtype
        assert torch.equal(y, y_ref), f"type {et} dtype {dt} shape {(H, I, n)}"


def test_switch_module_casts_weights_to_input_dtype():
    """expert_module.cpp:31-35: fp32 weights, bf16 activations -> weights are cast per call."""
    ws, x = rand_case(0, torch.float32, 64, 96, 6, 77)
    xb = x.to(torch.bfloat16)
    y_ref = LIVE["switch_cast"]
    assert y_ref.dtype == torch.bfloat16
    assert torch.equal(O.expert_ffn(xb, ws, 0), y_ref)
