"""Record what the reference itself computes for the tests that compare against it, so the comparisons run anywhere.

Run:  python tests/golden/make_reference_golden.py      (needs the reference tree; oracle/_ref built by __graft_entry__.build())
Writes
  expert_ffn_live_ref.pt   the compiled reference expert module (oracle/_ref/ref_expert_module.so) on the seeded random
                           shapes of tests/test_oracle_expert_ref.py;
  reference_results.pt     the literal reference Python (memory/*.py predictor, prefetcher, priority score; the
                           mixtral/deepseek/switch blocks), the compiled reference tensor-index code on the random stores of
                           tests/test_store_format.py, and the dispatch_local calls the literal blocks make
                           (tests/test_gpu_literal_blocks.py replays them on the GPU).
Every input is regenerated from its seed by the tests; what is stored is the reference's answer (and, where cheap, a
checksum of the inputs so that generator drift is caught).
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
for p in (ROOT, os.path.join(ROOT, "moe-infinity_b200"), TESTS, os.path.join(TESTS, "shims"), HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import make_golden as G  # noqa: E402
import ref_loader  # noqa: E402
import reference_cases as RC  # noqa: E402
from expert_cases import DT  # noqa: E402
from moe_infinity_b200.store import ArcherTensorStore  # noqa: E402
from oracle import ref_module  # noqa: E402


@contextlib.contextmanager
def _cpu_only_torch():
    """The literal ExpertTracer allocates on cuda:0 (expert_tracer.py:33-35,104); run it on CPU."""
    zeros, to = torch.zeros, torch.Tensor.to

    def zeros_cpu(*a, **k):
        k.pop("device", None)
        return zeros(*a, **k)

    def to_cpu(self, *a, **k):
        if any(isinstance(x, str) and x == "cpu" for x in a):
            return self.clone()      # cuda:0 -> cpu is a copy in the real run; keep that (the caller mutates it)
        a = tuple(x for x in a if not (isinstance(x, str) and x.startswith("cuda")))
        if not a and not k:
            return self
        return to(self, *a, **k)

    torch.zeros, torch.Tensor.to = zeros_cpu, to_cpu
    try:
        yield
    finally:
        torch.zeros, torch.Tensor.to = zeros, to


def _cfg(L, E):
    return types.SimpleNamespace(architectures=["MixtralForCausalLM"], num_hidden_layers=L, num_local_experts=E)


LIVE = os.path.join(HERE, "expert_ffn_live_ref.pt")
RESULTS = os.path.join(HERE, "reference_results.pt")
GPU_LITERAL_CASES = ["mixtral_mini_bf16", "mixtral_ragged_bf16", "mixtral_mini_f16", "mixtral_onetoken_bf16",
                     "deepseek_mini_bf16", "deepseek_group_bf16", "switch_mini_bf16", "nllb_mini_bf16", "nllb_capacity_f16"]


def expert_module(R):
    torch.set_num_threads(1)
    live = {}
    for et in range(6):
        for di in range(3):
            ys = []
            for i, (H, I, n) in enumerate(RC.SHAPES):
                ws, x = RC.rand_case(et, DT[di], H, I, n, RC.seed_of(et, di, i))
                ys.append(R.expert_forward(et, di, ws, x))
            live[(et, di)] = ys
    ws, x = RC.rand_case(0, torch.float32, 64, 96, 6, 77)
    live["switch_cast"] = R.expert_forward(0, 1, ws, x.to(torch.bfloat16))
    return live


def memory_policy(ns):
    """The literal ExpertTracer/ExpertPredictor, ExpertPrefetcher and priority_score on the tests' seeded inputs."""
    import importlib
    out = {"predictor": {}, "priority_score": {}}
    L, E, cap = 6, 8, 12
    for seed in RC.PREDICTOR_SEEDS:
        rng = np.random.default_rng(seed)
        lib = RC.library(rng, 9, L, E)
        with _cpu_only_torch():
            ns.expert_tracer.ExpertTracer._instance = None
            rt = ns.expert_tracer.ExpertTracer(cap, _cfg(L, E))
            rt.trace_collection[:9] = torch.from_numpy(lib)
            rp = ns.expert_predictor.ExpertPredictor(_cfg(L, E))
            rp.add_tracer(rt)
            rs = rt.create_entry()
            preds = []
            for step in range(3):
                for layer in range(L):
                    experts = rng.integers(0, E, size=(4, 2))
                    preds.append(np.asarray(rp.predict(rs, torch.from_numpy(experts), layer), dtype=np.float64))
            out["predictor"][seed] = dict(predict=np.stack(preds), matrix=np.asarray(rt.get_entry(rs).matrix),
                                          collection_access=np.asarray(rt.collection_access))
    L, E = 5, 4
    matrix, tmap = RC.prefetch_inputs(L, E)

    class Rec:
        def __init__(self):
            self.cands, self.enq = None, []

        def replace_cache_candidates(self, ids):
            self.cands = list(ids)

        def get_node_default_device(self, ids):
            return 0

        def enqueue_prefetch(self, tid, gpu):
            self.enq.append(tid)

    with contextlib.redirect_stdout(io.StringIO()):
        rp = ns.expert_prefetcher.ExpertPrefetcher(_cfg(L, E))
    rp.expert_tensor_map = tmap
    r = Rec()
    rp.set_archer_engine(r)
    rp.prefetch_experts(2, matrix)
    out["prefetch"] = dict(cands=[int(c) for c in r.cands], enq=[int(t) for t in r.enq])
    ps = importlib.import_module("moe_infinity.memory.expert_priority_score")
    ent = importlib.import_module("moe_infinity.memory.expert_entry")
    for current_layer in RC.PRIORITY_LAYERS:
        L, E, dec, freq = RC.priority_inputs(current_layer)
        entry = ent.ExpertTraceEntry("s", dec.copy(), 0, 0)
        ref_m = np.zeros((L, E))
        for ce in ps.priority_score(freq, set(), set(), entry, current_layer, L):
            ref_m[ce.layer_idx, ce.expert_idx] = ce.r
        out["priority_score"][current_layer] = ref_m
    return out


def literal_blocks(ns):
    """The literal blocks' outputs on the fixture cases that tests/test_oracle_golden.py holds the oracle to."""
    out = {}
    for name in ("mixtral_mini_bf16", "mixtral_ragged_bf16"):
        c = G.build_mixtral(name)
        l_out, l_logits = G.run_literal_mixtral(ns, c["H"], c["I"], c["E"], c["k"], c["hidden"], c["gate"], c["experts"])
        out[name] = dict(out=l_out, logits=l_logits)
    name = "deepseek_group_bf16"
    c = G.build_deepseek(name)
    out[name] = dict(out=G.run_literal_deepseek(ns, c["H"], c["I"], c["E"], c["k"], c["n_shared"], c["hidden"], c["gate"],
                                                c["experts"], c["shared"], c["topk_method"], c["n_group"], c["topk_group"],
                                                c["norm_topk_prob"], c["routed_scaling_factor"]))
    for name in G.SWITCH_CASES:
        c = G.build_switch(name)
        l_out, l_logits, l_index = G.run_literal_switch(ns, c["H"], c["I"], c["E"], c["capacity"], c["hidden"], c["gate"],
                                                        c["experts"])
        out[name] = dict(out=l_out, logits=l_logits, index=l_index)
    return out


class _Recorder:
    """Stands between a literal block and its expert executor; keeps the arguments of every dispatch_local call."""

    def __init__(self, inner, calls):
        self.inner, self.calls = inner, calls

    def dispatch_local(self, hidden_states, router_mask, layer_id):
        self.calls.append(dict(hidden=hidden_states.detach().clone(), router_mask=router_mask.detach().clone(),
                               layer_id=int(layer_id)))
        return self.inner.dispatch_local(hidden_states, router_mask, layer_id)


@contextlib.contextmanager
def _recording(calls):
    setattr_ = torch.nn.Module.__setattr__

    def rec_setattr(self, name, value):
        if name == "expert_executor":
            value = _Recorder(value, calls)
        setattr_(self, name, value)
    torch.nn.Module.__setattr__ = rec_setattr
    try:
        yield
    finally:
        torch.nn.Module.__setattr__ = setattr_


def dispatch_calls(ns):
    """dispatch_local calls of the literal blocks (CPU, the fixtures' inputs), per case of tests/test_gpu_literal_blocks.py."""
    out = {}
    for name in GPU_LITERAL_CASES:
        calls = []
        with _recording(calls):
            if name in G.MIXTRAL_CASES:
                c = G.build_mixtral(name)
                G.run_literal_mixtral(ns, c["H"], c["I"], c["E"], c["k"], c["hidden"], c["gate"], c["experts"])
            elif name in G.DEEPSEEK_CASES:
                c = G.build_deepseek(name)
                G.run_literal_deepseek(ns, c["H"], c["I"], c["E"], c["k"], c["n_shared"], c["hidden"], c["gate"], c["experts"],
                                       c["shared"], c["topk_method"], c["n_group"], c["topk_group"], c["norm_topk_prob"],
                                       c["routed_scaling_factor"])
            elif name in G.SWITCH_CASES:
                c = G.build_switch(name)
                G.run_literal_switch(ns, c["H"], c["I"], c["E"], c["capacity"], c["hidden"], c["gate"], c["experts"])
            else:
                c = G.build_nllb(name)
                G.run_literal_nllb(ns, c["H"], c["I"], c["E"], c["capacity"], c["hidden"], c["gate"], c["experts"])
        assert calls, name
        out[name] = calls
    return out


def store_index(R):
    """Per seed: our writer's index file, the reference reader's view of it, and the reference writer's file for the same
    metas."""
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for seed in RC.STORE_SEEDS:
            tensors = RC.random_tensors(seed, 25)
            d = os.path.join(tmp, f"s{seed}")
            store = ArcherTensorStore(d)
            for tid, t in tensors.items():
                store.store_tensor(tid, t, flush=False)
            store.flush()
            with open(store.index_path, "rb") as f:
                ours = f.read()
            deser = {int(e[0]): tuple(e[1:]) for e in R.index_deserialize(store.index_path)}
            ref_path = os.path.join(d, "ref_index")
            R.index_serialize(ref_path, [(tid, store.index[tid].file_id, store.index[tid].offset, t) for tid, t in tensors.items()])
            with open(ref_path, "rb") as f:
                ref_bytes = f.read()
            out[seed] = dict(our_index=ours, ref_deserialize=deser, ref_index=ref_bytes)
    return out


def main():
    R = ref_module.load()
    assert R is not None, "oracle/_ref/ref_expert_module.so missing (python __graft_entry__.py builds it)"
    assert ref_loader.available(), "reference Python tree not found"
    ns = ref_loader.load()
    torch.save(expert_module(R), LIVE)
    torch.save(dict(memory=memory_policy(ns), literal=literal_blocks(ns), dispatch_calls=dispatch_calls(ns), store=store_index(R)),
               RESULTS)
    for p in (LIVE, RESULTS):
        print(p, os.path.getsize(p), "bytes")


if __name__ == "__main__":
    main()
