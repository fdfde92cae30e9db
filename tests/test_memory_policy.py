"""CPU: host policy code -- tracer/predictor/prefetcher mirrors against what the LITERAL reference classes
(moe_infinity/memory/*.py of the reference) computed on the same seeded inputs (tests/golden/reference_results.pt, written by
tests/golden/make_reference_golden.py), and the cache-policy oracle's stated rules."""
import os

import numpy as np
import pytest
import torch

from moe_infinity_b200 import memory as M
from oracle.policy_oracle import CacheOracle
from reference_cases import PREDICTOR_SEEDS, PRIORITY_LAYERS, library, prefetch_inputs, priority_inputs

REF = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_results.pt"),
                 weights_only=False)["memory"]


@pytest.mark.parametrize("seed", PREDICTOR_SEEDS)
def test_predictor_matches_literal_reference(seed):
    ref = REF["predictor"][seed]
    L, E, cap = 6, 8, 12
    rng = np.random.default_rng(seed)
    lib = library(rng, 9, L, E)
    ot = M.ExpertTracer(cap, L, E)
    ot.load_trace(lib)
    op = M.ExpertPredictor(L, E)
    op.add_tracer(ot)
    os_ = ot.create_entry()
    i = 0
    for step in range(3):
        for layer in range(L):
            experts = rng.integers(0, E, size=(4, 2))
            b = op.predict(os_, experts, layer)
            np.testing.assert_allclose(ref["predict"][i], b, rtol=1e-6, atol=1e-9)
            i += 1
    assert i == len(ref["predict"])
    np.testing.assert_array_equal(ref["matrix"], ot.get_entry(os_).matrix)
    np.testing.assert_array_equal(ref["collection_access"], ot.collection_access)


def test_prefetch_request_order_matches_literal_reference():
    ref = REF["prefetch"]
    L, E = 5, 4
    matrix, tmap = prefetch_inputs(L, E)

    class Rec:
        def __init__(self):
            self.cands, self.enq = None, []

        def replace_cache_candidates(self, ids):
            self.cands = list(ids)

        def get_node_default_device(self, ids):
            return 0

        def enqueue_prefetch(self, tid, gpu):
            self.enq.append(tid)

    op = M.ExpertPrefetcher(L, E)
    op.expert_tensor_map = tmap
    r2 = Rec()
    op.set_archer_engine(r2)
    op.prefetch_experts(2, matrix)
    assert ref["cands"] == r2.cands and ref["enq"] == r2.enq
    assert [tmap[p] for p, _ in op.ordered_requests(2, matrix)] == ref["enq"]


def test_degenerate_empty_library_prefetches_everything_nearest_first():
    """SURVEY §9 Q8: with no trace library the predictor degenerates to 'all experts of later layers, nearest first'."""
    L, E = 4, 3
    tr = M.ExpertTracer(5, L, E)
    pr = M.ExpertPredictor(L, E)
    pr.add_tracer(tr)
    sid = tr.create_entry()
    m = pr.predict(sid, np.array([[0, 1]]), 1)
    assert np.all(m[0] == 0) and np.all(m[1:] > 0)
    pf = M.ExpertPrefetcher(L, E)
    reqs = pf.ordered_requests(1, m)
    assert [p[0] for p, _ in reqs] == [1] * E + [2] * E + [3] * E


def test_tracer_finish_entry_and_counts():
    tr = M.ExpertTracer(2, 3, 4)
    sid = tr.create_entry()
    tr.update_entry(sid, np.array([[1, 1], [2, 3]]), 0)
    assert tr.get_entry(sid).matrix[0].tolist() == [0, 2, 1, 1]
    tr.update_entry(sid, np.array([[0, 1]]), 2)
    assert tr.get_entry(sid).num_new_tokens == 1
    tr.finish_entry(sid)
    assert tr.trace_collection[0].sum() == 6 and tr.collection_access[0] == 1


@pytest.mark.parametrize("current_layer", PRIORITY_LAYERS)
def test_priority_score_matches_literal_reference(current_layer):
    L, E, dec, freq = priority_inputs(current_layer)
    ours = M.priority_score_matrix(freq, dec, current_layer, L)
    np.testing.assert_allclose(ours, REF["priority_score"][current_layer], rtol=1e-12, atol=0)


# ---------------------------------------------------------------- cache policy oracle: the stated rules
def test_cache_oracle_lfu_eviction_and_tie_order():
    c = CacheOracle(num_layers=2, num_experts=4, num_slots=3, policy="slots")
    assert c.dispatch(0, [0, 1]) == [(0, False), (1, False)]
    assert c.dispatch(0, [0]) == [(0, True)]                 # visits: (0,0)=2, (0,1)=1
    assert c.dispatch(1, [2]) == [(2, False)]                # third slot
    assert c.dispatch(1, [3]) == [(3, False)]                # evicts min visits, ties -> expert-major scan
    assert c.evicted_log == [(0, 1)]                         # (0,1) and (1,2) both have 1 visit; expert 1 scanned first
    assert c.stats["misses"] == 4 and c.stats["hits"] == 1
    # the reference's byte budget is charged for hits too (expert_dispatcher.cpp:266): after 2 misses + 1 hit the budget
    # of 3 experts is used up, so the third miss already evicts although a slot is physically free
    # (behaviour confirmed on the reference's real engine: tests/golden/policy_ref_trace.json never holds 9 of its 9 experts)
    r = CacheOracle(num_layers=2, num_experts=4, num_slots=3, policy="reference")
    r.dispatch(0, [0, 1]); r.dispatch(0, [0]); r.dispatch(1, [2]); r.dispatch(1, [3])
    assert r.evicted_log == [(0, 1), (1, 2)] and sum(r.resident) == 2


def test_cache_oracle_waves_when_active_set_exceeds_slots():
    c = CacheOracle(1, 4, 2)
    c.dispatch(0, [0, 1])
    # 3 active experts, 2 slots: wave 1 = {1 (hit)} + nothing else fits without evicting a still-to-run expert...
    res = c.dispatch(0, [1, 2, 3])
    assert res == [(1, True), (2, False), (3, False)]
    assert c.stats["evictions"] == 2 and sum(c.resident) == 2
    c0 = CacheOracle(1, 4, 0)
    with pytest.raises(RuntimeError):
        c0.dispatch(0, [0])


def test_cache_oracle_prefetch_respects_protection():
    c = CacheOracle(2, 4, 2)
    c.dispatch(0, [0, 1])
    c.prefetch_hint([(1, 0), (1, 1), (1, 2)], [0.9, 0.5, 0.7])
    # last dispatch is in use -> nothing evictable -> no prefetch
    assert c.stats["prefetch_issued"] == 0
    c.dispatch(1, [3])                  # evicts (0,0) [visits equal, expert-major]
    c.prefetch_hint([(0, 0)], [1.0])    # (0,1) evictable (not protected, not in use)
    assert c.stats["prefetch_issued"] == 1 and c.evicted_log[-1] == (0, 1)
    c.prefetch_hint([(0, 0), (0, 2)], [1.0, 0.5])   # (0,0) resident+protected; (1,3) in use -> (0,2) dropped
    assert c.stats["prefetch_issued"] == 1
    assert c.dispatch(0, [0]) == [(0, True)] and c.stats["prefetch_useful"] == 1
