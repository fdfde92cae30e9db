"""CPU: the oracle against the committed golden vectors, and against what the literal reference block files computed on the
same inputs (tests/golden/reference_results.pt, written by tests/golden/make_reference_golden.py)."""
import os

import pytest
import torch

from oracle import moe_oracle as O
import make_golden as G

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LITERAL = torch.load(os.path.join(GOLDEN, "reference_results.pt"), weights_only=False)["literal"]


def _load(name):
    return torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)


@pytest.mark.parametrize("name", list(G.MIXTRAL_CASES))
def test_mixtral_oracle_matches_golden(name):
    fx = _load(name)
    c = G.build_mixtral(name)
    assert abs(G.checksum([w for e in c["experts"] for w in e]) - fx["weight_checksum"]) <= 1e-6 * fx["weight_checksum"]
    out, logits, r = O.mixtral_block(c["hidden"], c["gate"], c["experts"], c["k"])
    assert torch.equal(logits, fx["router_logits"])
    assert torch.equal(r.topk_idx, fx["topk_idx"])
    assert torch.equal(r.topk_weight, fx["topk_weight"])
    ok = ~fx["tied"]
    assert torch.equal(out.reshape(-1, c["H"])[ok], fx["out"].reshape(-1, c["H"])[ok])
    y32 = O.combine_fp32(c["hidden"], c["experts"], r.topk_idx, r.topk_weight, O.MIXTRAL_MOE_DENSE_ACT_DENSE)
    assert torch.allclose(y32, fx["out_fp32"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("name", list(G.DEEPSEEK_CASES))
def test_deepseek_oracle_matches_golden(name):
    fx = _load(name)
    c = G.build_deepseek(name)
    kw = {k: c[k] for k in ("topk_method", "n_group", "topk_group", "norm_topk_prob", "routed_scaling_factor")}
    out, r = O.deepseek_block(c["hidden"], c["gate"], c["experts"], c["k"], c["shared"], **kw)
    assert torch.equal(r.scores, fx["scores"])
    assert torch.equal(r.topk_idx, fx["topk_idx"])
    ok = ~fx["tied"]
    a, b = out.reshape(-1, c["H"])[ok], fx["out"].reshape(-1, c["H"])[ok]
    assert torch.equal(a, b)


@pytest.mark.parametrize("name", list(G.SWITCH_CASES))
def test_switch_oracle_matches_golden(name):
    fx = _load(name)
    c = G.build_switch(name)
    out, (logits, idx), mask = O.switch_block(c["hidden"], c["gate"], c["experts"], c["capacity"])
    assert torch.equal(out, fx["out"]) and torch.equal(mask, fx["router_mask"])
    # capacity: no expert holds more than `capacity` tokens of one batch row
    assert int(mask.sum(dim=1).max()) <= c["capacity"]


def test_topk_tie_break_lowest_index():
    s = torch.tensor([[0.2, 0.3, 0.3, 0.2], [0.25, 0.25, 0.25, 0.25]])
    v, i = O.topk_lowest_index(s, 2)
    assert i.tolist() == [[1, 2], [0, 1]]
    assert O.tied_tokens(s, 2).tolist() == [False, True]
    assert O.tied_tokens(s, 1).tolist() == [True, True]


def test_mixtral_masks_match_one_hot_definition():
    torch.manual_seed(0)
    logits = torch.randn(50, 8).to(torch.bfloat16)
    r = O.mixtral_route(logits, 2, torch.bfloat16)
    assert r.router_mask.dtype == torch.bool and r.router_mask.sum(-1).eq(2).all()
    w = torch.zeros(50, 8, dtype=torch.bfloat16).scatter_(1, r.topk_idx, r.topk_weight)
    assert torch.equal(w, r.routing_weights_mask)


def test_empty_and_single_expert_edge_cases():
    experts = O.make_experts(4, 64, 128, torch.bfloat16, 1)
    x = torch.zeros(1, 0, 64, dtype=torch.bfloat16)
    out, logits, r = O.mixtral_block(x, torch.zeros(4, 64, dtype=torch.bfloat16), experts, 2)
    assert out.shape == (1, 0, 64)
    # all tokens to the same two experts (constant logits -> ties -> experts 0,1)
    x = torch.randn(1, 5, 64).to(torch.bfloat16)
    out, logits, r = O.mixtral_block(x, torch.zeros(4, 64, dtype=torch.bfloat16), experts, 2)
    assert r.topk_idx.tolist() == [[0, 1]] * 5 and O.tied_tokens(r.scores, 2).all()


@pytest.mark.parametrize("name", ["mixtral_mini_bf16", "mixtral_ragged_bf16"])
def test_literal_reference_block_equals_oracle(name):
    c = G.build_mixtral(name)
    l_out, l_logits = LITERAL[name]["out"], LITERAL[name]["logits"]
    o_out, o_logits, r = O.mixtral_block(c["hidden"], c["gate"], c["experts"], c["k"])
    assert torch.equal(l_logits, o_logits)
    ok = ~O.tied_tokens(r.scores, c["k"])
    assert torch.equal(l_out.reshape(-1, c["H"])[ok], o_out.reshape(-1, c["H"])[ok])


def test_literal_deepseek_block_equals_oracle():
    name = "deepseek_group_bf16"
    c = G.build_deepseek(name)
    l_out = LITERAL[name]["out"]
    kw = {k: c[k] for k in ("topk_method", "n_group", "topk_group", "norm_topk_prob", "routed_scaling_factor")}
    o_out, r = O.deepseek_block(c["hidden"], c["gate"], c["experts"], c["k"], c["shared"], **kw)
    ok = ~O.tied_tokens(r.scores, c["k"])
    assert torch.equal(l_out.reshape(-1, c["H"])[ok], o_out.reshape(-1, c["H"])[ok])


@pytest.mark.parametrize("name", list(G.SWITCH_CASES))
def test_literal_switch_block_equals_oracle(name):
    """A6 pin: the reference's own SyncSwitchTransformersSparseMLP (switch_transformers.py:41-113) on the 4.x-order router
    shim, bit for bit against the oracle -- outputs, router logits, expert index, including capacity drops."""
    c = G.build_switch(name)
    l_out, l_logits, l_index = LITERAL[name]["out"], LITERAL[name]["logits"], LITERAL[name]["index"]
    o_out, (o_logits, o_index), mask = O.switch_block(c["hidden"], c["gate"], c["experts"], c["capacity"])
    assert torch.equal(l_logits.float(), o_logits.float())
    assert torch.equal(l_index, o_index)
    assert torch.equal(l_out, o_out)
    fx = _load(name)
    assert fx["source"] == "literal" and torch.equal(fx["out"], l_out)


@pytest.mark.parametrize("name", list(G.NLLB_CASES))
def test_literal_nllb_block_reproduces_its_golden(name):
    """The committed fixture is the output of the reference's own SyncNllbMoeSparseMLP (nllb_moe.py:20-115; HF's top-2 router
    on its 4.x contract) with the oracle's NllbMoeDenseActDense behind dispatch_local; that output is the literal combine of
    the oracle's per-expert results (the part a plugin must get right)."""
    c = G.build_nllb(name)
    fx = _load(name)
    assert fx["kind"] == "nllb" and fx["source"] == "literal" and torch.equal(fx["hidden"], c["hidden"])
    assert abs(G.checksum([w for e in c["experts"] for w in e]) - fx["weight_checksum"]) <= 1e-6 * fx["weight_checksum"]
    out, probs = fx["out"], fx["router_probs"]
    # restated combine: per expert, weights * output added in ascending expert order; untouched elements keep the input
    x = c["hidden"].reshape(-1, c["H"])
    w = probs.reshape(-1, c["E"])
    acc = torch.zeros_like(x)
    for o, _, e, _ in O.dispatch_local(x, w.bool(), c["experts"], O.NLLB_MOE_DENSE_ACT_DENSE):
        idx = w[:, e].bool()
        acc[idx] += torch.einsum("b,be->be", w[idx, e], o)
    acc[acc == 0] = x[acc == 0]
    assert torch.equal(acc.reshape(out.shape), out)
    n = w.bool().sum(-1)
    assert int(n.max()) == 2 and (name != "nllb_capacity_f16" or int(n.min()) < 2)      # the capacity case really drops
