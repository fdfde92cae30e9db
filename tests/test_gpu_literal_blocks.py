"""GPU: the calls the reference's OWN, unmodified MoE blocks (moe_infinity/models/{mixtral,deepseek,switch_transformers,nllb_moe}.py)
make into their expert executor, replayed on a B200 into this repository's plugin objects, constructed exactly the way
moe_infinity/runtime/model_offload.py constructs the reference's (`prefetch_handle(prefix, ratio)`,
`expert_dispatcher(E, L, dtype, expert_type, num_threads)` -- five positional arguments, :143-145, :471-477 -- then
`offload` / `register_expert` / `set_expert_dispatcher`).  The literal blocks ran on CPU on the fixtures' inputs
(tests/golden/make_reference_golden.py); every `expert_executor.dispatch_local(hidden_states, router_mask, layer_id)` they
issued -- 2-D or 3-D hidden states, the masks exactly as the block built them -- is stored in tests/golden/reference_results.pt.
Everything behind `dispatch_local` is libb2m.so; each returned expert output is held to the oracle's, which
tests/test_oracle_golden.py and tests/test_oracle_expert_ref.py pin bit for bit to the literal blocks and the reference's
compiled expert module."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import moe_oracle as O  # noqa: E402
from test_gpu_parity import hidden_close, load_case  # noqa: E402

CALLS = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_results.pt"),
                   weights_only=False)["dispatch_calls"]


def _plugin(c, expert_type, dtype_int, layers=1):
    """The three objects OffloadEngine builds (model_offload.py:143-160, 471-477), reference signatures only."""
    from moe_infinity_b200.compat import DistributedExpertExecutor, expert_dispatcher, prefetch_handle
    h = prefetch_handle("/tmp/b2m_literal_unused", 0.9)
    d = expert_dispatcher(c["E"], layers, dtype_int, expert_type, 8)
    assert d.handle is h
    tid = 0
    for e in range(c["E"]):
        ids = []
        for w in c["experts"][e]:                      # named_parameters order
            h.offload(w, tid)
            ids.append(tid)
            tid += 1
        d.register_expert(0, e, ids)                   # model_offload.py:851-853
    ex = DistributedExpertExecutor()
    ex.set_expert_dispatcher(d)
    return h, d, ex


def _replay(name, c, expert_type, dtype_int):
    """Every recorded dispatch_local call of the literal block, through the plugin on the GPU, against the oracle."""
    _, d, ex = _plugin(c, expert_type, dtype_int)
    dt = c["dtype"]
    calls = CALLS[name]
    assert calls
    for call in calls:
        hidden, mask, lid = call["hidden"], call["router_mask"], call["layer_id"]
        assert hidden.dtype == dt and mask.shape[-1] == c["E"]
        with torch.no_grad():
            got = ex.dispatch_local(hidden.cuda(), mask.cuda(), lid)
        torch.cuda.synchronize()
        want = O.dispatch_local(hidden, mask, c["experts"], expert_type, lid)
        assert [(l, e) for _, l, e, _ in got] == [(l, e) for _, l, e, _ in want], "experts returned differ"
        for (y, _, e, _), (y_ref, _, _, _) in zip(got, want):
            assert y.is_cuda and y.dtype == dt and y.shape == y_ref.shape
            hidden_close(y, y_ref, None, dt, f"literal {name} call, expert {e}")
    return d


@pytest.mark.parametrize("name", ["mixtral_mini_bf16", "mixtral_ragged_bf16", "mixtral_mini_f16", "mixtral_onetoken_bf16"])
def test_literal_mixtral_block_on_gpu(lib_built, name):
    from moe_infinity_b200 import _lib as L
    c, _ = load_case(name)
    d = _replay(name, c, L.EXPERT_MIXTRAL, L.DTYPE_BF16 if c["dtype"] == torch.bfloat16 else L.DTYPE_F16)
    assert d.engine.k == c["k"]                         # top_k learnt from the masks


@pytest.mark.parametrize("name", ["deepseek_mini_bf16", "deepseek_group_bf16"])
def test_literal_deepseek_block_on_gpu(lib_built, name):
    """deepseek.py:8-137 with the literal MoEGate: top-k 4 masks reach a dispatcher that was built without a top_k."""
    from moe_infinity_b200 import _lib as L
    c, _ = load_case(name)
    d = _replay(name, c, L.EXPERT_DEEPSEEK, L.DTYPE_BF16)
    assert d.engine.k >= c["k"]


@pytest.mark.parametrize("name", ["switch_mini_bf16"])
def test_literal_switch_block_on_gpu(lib_built, name):
    """switch_transformers.py:41-113 on the 4.x-order router shim: 3-D hidden states and one-hot masks."""
    from moe_infinity_b200 import _lib as L
    c, _ = load_case(name)
    _replay(name, c, L.EXPERT_SWITCH, L.DTYPE_BF16)


@pytest.mark.parametrize("name", ["nllb_mini_bf16", "nllb_capacity_f16"])
def test_literal_nllb_block_on_gpu(lib_built, name):
    """nllb_moe.py:20-115 (HF top-2 router on its 4.x contract, 3-D hidden states and masks handed to dispatch_local, bias
    experts fc1|fc1_bias|fc2|fc2_bias, tokens dropped by the router's capacity in no mask column)."""
    import make_golden as G
    from moe_infinity_b200 import _lib as L
    fx = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".pt"), weights_only=False)
    c = G.build_nllb(name)
    assert torch.equal(c["hidden"], fx["hidden"])
    _replay(name, c, L.EXPERT_NLLB, L.DTYPE_BF16 if c["dtype"] == torch.bfloat16 else L.DTYPE_F16)
