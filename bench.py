#!/usr/bin/env python
"""bench.py -- decode tokens/s + p50 per-token latency of the MoE dispatch hot path, Mixtral-8x7B shapes.

Usage: `python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]`
prints ONE JSON line on rank 0.  --dump-outputs DIR (single-GPU Mixtral path) writes DIR/out.npy: the float32 copy of the
[layers, 8, 4096] hidden states the last timed step returned; the inputs are seeded, so two builds can be compared output for
output.  Nothing is written into the source tree.

Workload (N=1, BASELINE.json configs[1]): Mixtral-8x7B bf16, random-init N(0,0.02^2) weights, 32 MoE layers,
8 experts, top-2, H=4096, I=14336; decode batch 8 => T=8 tokens enter every MoE block per step; all 256
experts HBM resident (90.2 GB).  A "step" = one pass of the hot path (router gate + softmax/top-k + permute +
grouped gate/up GEMM with fused SwiGLU + grouped down GEMM + weighted combine) over the 32 layers for one batch
of synthetic hidden states (the attention between MoE blocks is outside the path, SURVEY §8).
  value : whole-job tokens/s with inputs resident in HBM, the 32-layer step replayed as one CUDA graph.
  e2e   : same metric through the public Python API with HOST buffers (DecodeSession.step()): the step's inputs
          are copied from pinned host memory and its outputs copied back inside the timed region; the per-layer
          eager API (MoEEngine.forward x 32) is reported next to it.
  roofline : dominant kernel = grouped gate/up GEMM (K3, 2/3 of the weight bytes), timed with CUDA events on
          its launch stream; algorithmic bytes counted from the actual routing of the timed inputs.
  cpu_baseline : the reference's CPU path on the host cores for a bounded sample (as many full-size layers as fit
          ~12 s): routing/combine restated from mixtral.py, expert FFN = the reference's own compiled
          core/parallel/expert_module.cpp (oracle/_ref/ref_expert_module.so, kind "reference"; the oracle port if
          that .so is absent), at the fastest thread count of a sweep -- also used as a full-size parity check.
--impl reference times that CPU path alone (the reference's complete native engine needs a GPU: its GPU-side
timing is tools/ref_engine_harness.py, profiles/r02_ref_engine.json).
N>1: expert parallel over N ranks (rank r owns experts [r*E/N, (r+1)*E/N)), weak scaling (batch 8 per rank),
fused peer-to-peer token dispatch over NVLink (B2M_EP_EXCHANGE=nccl selects the NCCL all-to-all baseline);
see moe_infinity_b200/ep.py.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True          # the tree may be read-only: no __pycache__ next to the sources
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "moe-infinity_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

MIXTRAL = dict(L=32, E=8, H=4096, I=14336, k=2)
BATCH = 8
METRIC = "decode tokens/sec + p50 per-token latency, Mixtral-8x7B MoE dispatch path"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel (K3), from the newest COMMITTED
    `ncu --set full` capture of this command -- a property of that capture (one layer with 7 activated experts), not of the run
    that prints it: returned together with its source so the JSON line says so.  None if no capture is committed."""
    for name in ("r02b_dram_traffic.json", "r01k_dram_traffic.json", "r01_k3_dram_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            with open(path) as f:
                d = json.load(f)
            return d.get("traffic_bytes_per_launch"), f"profiles/{name}: {d.get('source', 'ncu --set full capture')}"
    return None, None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_layer_fn():
    """One MoE layer of the reference's path on the host: routing + mask build + combine as moe_infinity/models/mixtral.py:44-101
    states them (oracle restatement), expert FFN = the reference's OWN compiled module (oracle/_ref/ref_expert_module.so =
    core/parallel/expert_module.cpp built as-is, kind "reference") when it travelled with the snapshot, else the oracle's
    op-for-op port of it (kind "port", pinned bit-for-bit to the same module by tests/test_oracle_expert_ref.py)."""
    import torch.nn.functional as F
    from oracle import moe_oracle as O
    from oracle import ref_module
    ref = None
    try:
        ref = ref_module.load()
    except Exception:
        ref = None

    def layer(x, gate, experts, k):
        Hh = x.shape[-1]
        x2 = x.reshape(-1, Hh)
        logits = F.linear(x2, gate)                                    # mixtral.py:46
        r = O.mixtral_route(logits, k, x2.dtype)                       # :48-65
        final = torch.zeros_like(x2)                                   # :87-91
        for e in range(len(experts)):                                  # dispatch_local + combine, ascending expert id
            idx = r.router_mask[:, e].bool()
            if not bool(idx.any()):
                continue
            xe = x2[idx]
            y = ref.expert_forward(O.MIXTRAL_MOE_DENSE_ACT_DENSE, 0, list(experts[e]), xe) if ref is not None \
                else O.expert_ffn(xe, experts[e], O.MIXTRAL_MOE_DENSE_ACT_DENSE)
            final[idx] += y * r.routing_weights_mask[idx, e][:, None]  # :96-101
        return final, logits, r
    return layer, ("reference" if ref is not None else "port")


def pick_cpu_threads(layer, x, gate, experts, k):
    """The fastest torch thread count for this box and this shape (T=8 rows against 117 MB matrices is bandwidth bound and
    bf16 matmul paths differ per CPU: round 1 measured 64 threads 3x SLOWER than 1).  Sweep, keep the best, say which."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (1, 4, 8, 16, 24, 32, 48, 64, ncpu) if c <= ncpu})
    best, best_t, table = 1, None, {}
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            layer(x, gate, experts, k)                      # warm (thread pool, page faults)
            dt = None
            for _ in range(2):                              # best of two: one sample per candidate was too noisy
                t0 = time.perf_counter()
                layer(x, gate, experts, k)
                el = time.perf_counter() - t0
                dt = el if dt is None else min(dt, el)
                if el > 1.0:
                    break
            table[c] = round(dt, 4)
            if best_t is None or dt < best_t:
                best, best_t = c, dt
            if dt > 4 * best_t and dt > 2.0:                # hopeless direction: stop burning the budget
                break
    # the single-shot sweep is noisy (a 48-thread sample once looked best and then ran 3x slower): re-time the three best
    # candidates with three repetitions each and keep the best median
    finalists = sorted(table, key=lambda c: table[c])[:3]
    med = {}
    with torch.no_grad():
        for c in finalists:
            torch.set_num_threads(c)
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                layer(x, gate, experts, k)
                ts.append(time.perf_counter() - t0)
            med[c] = sorted(ts)[1]
    best = min(med, key=lambda c: med[c])
    best_t = med[best]
    table = dict(table, **{f"median3@{c}": round(v, 4) for c, v in med.items()})
    torch.set_num_threads(best)
    return best, best_t, table


def make_cpu_layer(E, H, I, dtype, seed):
    """Full-size layer weights on the host.  randn on 1.4 G elements is slow on CPU, so draw uniform blocks with
    matching variance (std 0.02) -- the CPU baseline only needs realistic sizes/values, not a named checkpoint."""
    g = torch.Generator().manual_seed(seed)
    experts = []
    a = 0.02 * (3 ** 0.5)
    for _ in range(E):
        ws = []
        for shape in ((I, H), (H, I), (I, H)):
            w = torch.empty(shape, dtype=torch.float32).uniform_(-a, a, generator=g).to(dtype)
            ws.append(w)
        experts.append(ws)
    return experts


def cpu_sample(layer, xs, gate, experts, k, budget_s, L_model):
    """Time `n` consecutive full-size layers (fresh inputs per layer, same 2.8 GB of weights: larger than any host cache)
    as one sample of a decode step; n = as many of the model's layers as fit the budget.  -> (sec per 32-layer step, n, reps)"""
    with torch.no_grad():
        t0 = time.perf_counter()
        layer(xs[0], gate, experts, k)
        t_layer = time.perf_counter() - t0
        n = int(max(1, min(L_model, budget_s / max(t_layer, 1e-6))))
        reps, times = 0, []
        t_all = time.perf_counter()
        while True:
            t0 = time.perf_counter()
            for l in range(n):
                layer(xs[l % len(xs)], gate, experts, k)
            times.append((time.perf_counter() - t0) * L_model / n)
            reps += 1
            if time.perf_counter() - t_all >= budget_s or reps >= 3:
                break
    return sum(times) / len(times), n, reps


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores.  Each step = as many of
    the 32 full-size layers as fit the time budget (all 32 when the box is fast enough), scaled to 32; said in `config`."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = MIXTRAL
    dtype = torch.bfloat16
    layer, kind = cpu_reference_layer_fn()
    experts = make_cpu_layer(cfg["E"], cfg["H"], cfg["I"], dtype, 1234)
    g = torch.Generator().manual_seed(7)
    gate = (torch.randn(cfg["E"], cfg["H"], generator=g) * 0.02).to(dtype)
    # the arm's workload at N GPUs is the GPU arm's: weak scaling, batch 8 per GPU -> 8*N tokens per step through every layer
    T = BATCH * max(1, args.gpus)
    xs = [torch.randn(1, T, cfg["H"], generator=g).to(dtype) for _ in range(cfg["L"])]
    threads, t_layer, table = pick_cpu_threads(layer, xs[0], gate, experts, cfg["k"])
    # bound the whole run (steps + warm-up) to ~150 s: layers per timed step
    nrun = args.steps + max(1, args.warmup // 3)
    n_layers = int(max(1, min(cfg["L"], 150.0 / nrun / max(t_layer, 1e-6))))
    with torch.no_grad():
        for _ in range(max(1, args.warmup // 3)):
            for l in range(n_layers):
                layer(xs[l], gate, experts, cfg["k"])
        times = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            for l in range(n_layers):
                layer(xs[l], gate, experts, cfg["k"])
            times.append((time.perf_counter() - t0) * cfg["L"] / n_layers)
    step_s = sum(times) / len(times)
    value = T / step_s
    what = (f"every step = the {cfg['L']} full-size layers" if n_layers == cfg["L"] else
            f"every step = {n_layers} of the {cfg['L']} full-size layers, scaled x{cfg['L']}/{n_layers}")
    sample = (f"{args.steps} steps x {n_layers} full-size Mixtral layers (2.8 GB bf16 weights each pass, T={T}) on {threads} "
              f"threads of {os.cpu_count()} (thread sweep s/layer: {table})")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "p50_token_latency_ms": sorted(times)[len(times) // 2] * 1e3,
        "config": {"workload": f"Mixtral-8x7B MoE dispatch path, decode batch 8 per GPU x {max(1, args.gpus)} (T={T}), bf16, 32 layers x 8 "
                               "experts top-2, H=4096 I=14336; the reference's CPU path (routing/combine restated from mixtral.py, expert "
                               f"FFN kind '{kind}'); {what}", "inputs": "host memory", "global_batch": T,
                   "layers": cfg["L"], "layers_timed_per_step": n_layers, "threads": threads},
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def algorithmic_bytes(counts_per_layer, T, cfg):
    """SURVEY §8(d): per layer A*3*H*I*2 (weights of distinct activated experts) + 2*T*H*2 + T*E*2 + T*k*8."""
    H, I, E, k = cfg["H"], cfg["I"], cfg["E"], cfg["k"]
    total, k3 = 0, 0
    for c in counts_per_layer:
        A = sum(1 for v in c if v > 0)
        total += A * 3 * H * I * 2 + 2 * T * H * 2 + T * E * 2 + T * k * 8
        k3 += A * 2 * H * I * 2 + T * k * H * 2 + T * k * I * 2   # gate+up weights, gathered rows in, h out
    return total, k3


def dump_outputs(directory, **arrays):
    """What the timed path returned in its last step, as float32 .npy files (one per name)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


def run_ours(args):
    import torch.distributed as dist
    from moe_infinity_b200 import MoEEngine
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        from moe_infinity_b200 import ep
        return ep.bench_ep(args, MIXTRAL, BATCH, METRIC, load_peaks, ClockSampler)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cfg = dict(MIXTRAL)
    if args.layers:
        cfg["L"] = args.layers
    L, E, H, I, k = cfg["L"], cfg["E"], cfg["H"], cfg["I"], cfg["k"]
    T = BATCH
    dtype = torch.bfloat16
    t_setup = time.perf_counter()
    eng = MoEEngine(num_layers=L, num_experts=E, hidden=H, inter=I, top_k=k, dtype=dtype, max_tokens=max(T, 16),
                    num_slots=L * E)
    torch.manual_seed(0)
    for l in range(L):
        for e in range(E):
            v = eng.load_expert(l, e)            # flat bf16 view of the HBM slot
            v.normal_(0.0, 0.02)
        eng.set_gate(l, torch.randn(E, H, device=dev) * 0.02)
    x_dev = torch.randn(L, T, H, device=dev).to(dtype)
    out_dev = torch.empty_like(x_dev)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_setup

    def step_device():
        for l in range(L):
            eng.forward(l, x_dev[l], out=out_dev[l])

    # ---- eager warm-up (also sets kernel attributes outside of graph capture)
    for _ in range(2):
        step_device()
    torch.cuda.synchronize()
    launches0 = eng.stats()["kernel_launches"]
    step_device()
    launches_per_step = eng.stats()["kernel_launches"] - launches0
    # routing actually taken by the timed inputs -> algorithmic bytes
    counts = []
    for l in range(L):
        eng.route(l, x_dev[l])
        counts.append(eng.ws("counts", T).cpu().tolist())
    bytes_step, bytes_k3_step = algorithmic_bytes(counts, T, cfg)
    # ---- CUDA graph of one 32-layer step
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step_device()
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(graph):
        step_device()
    for _ in range(args.warmup):
        graph.replay()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    torch.cuda.synchronize()
    evs[0].record()
    for i in range(args.steps):
        graph.replay()
        evs[i + 1].record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out=out_dev)
    step_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    total_ms = evs[0].elapsed_time(evs[-1])
    ms_per_step = total_ms / args.steps
    value = BATCH * args.steps / (total_ms * 1e-3)
    p50 = sorted(step_ms)[len(step_ms) // 2]

    # ---- dominant kernel (K3) timed on its launch stream with CUDA events
    st = torch.cuda.current_stream()
    k3_ms = []
    for it in range(3 + min(args.steps, 10)):
        acc = 0.0
        for l in range(L):
            eng.route(l, x_dev[l])
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            eng.run_experts(l, T, phases=1)
            b.record(st)
            eng.run_experts(l, T, phases=2)
            eng.combine(l, x_dev[l], out=out_dev[l])
            b.synchronize()
            acc += a.elapsed_time(b)
        if it >= 3:
            k3_ms.append(acc / L)
    k3_avg_ms = sum(k3_ms) / len(k3_ms)
    peak, peak_src = load_peaks()
    k3_bytes = bytes_k3_step / L
    achieved = k3_bytes / (k3_avg_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "grouped_gemm_tc_kernel<16,dual> (gate/up + SwiGLU, K3)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": peak_src, "avg_launch_ms": k3_avg_ms, "algorithmic_bytes_per_launch": k3_bytes,
                "traffic": load_traffic()[0], "traffic_source": load_traffic()[1],
                "step": {"algorithmic_bytes": bytes_step, "achieved": bytes_step / (ms_per_step * 1e-3) / 1e9,
                         "frac": bytes_step / (ms_per_step * 1e-3) / 1e9 / peak}}

    # ---- e2e: public API with HOST buffers -- DecodeSession.step(): pinned host -> device copy of the step's inputs,
    # all 32 layers, device -> pinned host copy of the outputs, one stream synchronise; all inside the timed region
    from moe_infinity_b200 import DecodeSession
    sess = DecodeSession(eng, T).capture()
    sess.x_host.copy_(x_dev.cpu())
    for _ in range(max(3, args.warmup // 2)):
        sess.step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sess.step()
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    e2e_ms = max(e0.elapsed_time(e1), wall * 1e3)
    # same thing without the graph: MoEEngine.forward called layer by layer from Python
    x_host, out_host = sess.x_host, sess.out_host
    x_in = torch.empty_like(x_dev)

    def step_eager():
        x_in.copy_(x_host, non_blocking=True)
        for l in range(L):
            eng.forward(l, x_in[l], out=out_dev[l])
        out_host.copy_(out_dev, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(3):
        step_eager()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_eager()
    eager_ms = (time.perf_counter() - t0) * 1e3
    e2e = {"value": BATCH * args.steps / (e2e_ms * 1e-3), "unit": "tokens/s",
           "h2d_bytes_per_step": x_host.numel() * 2, "d2h_bytes_per_step": out_host.numel() * 2,
           "ms_per_step": e2e_ms / args.steps,
           "api": "DecodeSession.step(): graph of H2D copy + 32 x b2m_moe_forward + D2H copy, host synchronised",
           "eager_per_layer_api": {"value": BATCH * args.steps / (eager_ms * 1e-3), "ms_per_step": eager_ms / args.steps,
                                   "api": "MoEEngine.forward per layer (ctypes -> b2m_moe_forward)"}}

    # ---- cpu baseline on a bounded sample + full-size parity of layer 0
    cpu = None
    parity = None
    if not args.no_cpu:
        w0 = []
        for e in range(E):
            flat = eng.expert_device_view(0, e).cpu()
            m = H * I
            w0.append([flat[0:m].view(I, H), flat[m:2 * m].view(H, I), flat[2 * m:3 * m].view(I, H)])
        gate0 = eng._gates[0].cpu()
        x0 = x_dev[0].cpu().unsqueeze(0)
        layer_fn, kind = cpu_reference_layer_fn()
        threads, _, table = pick_cpu_threads(layer_fn, x0, gate0, w0, k)
        xs = [x_dev[l].cpu().unsqueeze(0) for l in range(L)]
        sec_step, n_l, reps = cpu_sample(layer_fn, xs, gate0, w0, k, args.cpu_seconds, L)
        with torch.no_grad():
            ref_out, ref_logits, r = layer_fn(x0, gate0, w0, k)
        cpu = {"value": BATCH / sec_step, "unit": "tokens/s", "cores": threads, "kind": kind,
               "sample": f"{reps} x {n_l} full-size layers (8 experts x 352 MB bf16, T=8) on {threads} threads of "
                         f"{os.cpu_count()}, scaled to {L} layers (thread sweep s/layer: {table})"}
        # full-size parity: same weights, same inputs, router logits from the oracle
        got = eng.forward(0, x_dev[0], router_logits=ref_logits.to(dev)).float().cpu()
        idx = eng.ws("topk_idx", T).cpu().long()
        ref = ref_out.reshape(T, H).float()
        rms = ref.pow(2).mean().sqrt().item()
        parity = {"expert_index_equal": bool(torch.equal(idx, r.topk_idx)),
                  "max_abs_diff": (got - ref).abs().max().item(), "ref_rms": rms,
                  "frac_bit_identical": (got == ref).float().mean().item()}

    line = {
        "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "p50_token_latency_ms": p50, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"Mixtral-8x7B MoE dispatch path, decode batch {BATCH} (T={T} tokens/layer/step), "
                               f"{L} layers x 8 experts top-2, H=4096 I=14336, bf16 random-init, all {L*E} experts "
                               f"HBM-resident ({L*E*3*H*I*2/1e9:.1f} GB); context 2048 affects attention only "
                               "(outside the path)",
                   "global_batch": BATCH, "layers": L, "parallelism": "single GPU",
                   "l2": "inputs larger than L2: each step streams ~%.1f GB of distinct expert weights" % (bytes_step / 1e9),
                   "numerics": "reference rounding chain", "timed_region": "CUDA graph replay of the 32-layer step"},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches_per_step * args.steps),
        "launches_per_step": int(launches_per_step), "clocks": clocks, "full_size_parity_layer0": parity,
        "setup_s": setup_s,
    }
    print(json.dumps(line), flush=True)


def run_offload(args):
    """--config offload = BASELINE configs[2]: Mixtral-8x7B bf16, device_memory_ratio 0.25 (forced offload), 32 layers, decode
    batch 8 on the SURVEY 8(d) trace: per-layer Zipf-1 popular experts (router bias folded into the gate weight through a
    constant hidden coordinate), hidden states AR(1) over decode steps (0.9) and over layers (0.9, the residual stream);
    one T=16384 prefill first.  All 256 experts live in pinned host DRAM (90 GB); HBM holds ratio x total / 352 MB of them.
    Two runs on the same trace: the reference's policy (on-demand fetch, evict min incache_visit_count,
    expert_dispatcher.cpp:227-266; prefetch off as on the reference's Mixtral block) and ours (activation-aware cache +
    router-logit look-ahead prefetch).  The step is bound by the host->device link: roofline = H2D bytes / time vs the
    pinned-copy bandwidth measured in the same process."""
    import ctypes as C
    from moe_infinity_b200 import MoEEngine, _lib as L_
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    cfg = dict(MIXTRAL)
    if args.layers:
        cfg["L"] = args.layers
    L, E, H, I, k = cfg["L"], cfg["E"], cfg["H"], cfg["I"], cfg["k"]
    T, dtype = BATCH, torch.bfloat16
    steps, warm = args.steps, max(2, args.warmup)
    ratio = args.ratio
    # ---- measured link peak
    nb = 1 << 30
    hb = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
    db = torch.empty(nb, dtype=torch.uint8, device=dev)
    for _ in range(2):
        db.copy_(hb, non_blocking=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(4):
        db.copy_(hb, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    h2d_peak = 4 * nb / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del hb, db
    # ---- host weights: 256 pinned blobs (values from one seeded draw, per-expert offset so experts differ)
    t0 = time.perf_counter()
    nel = 3 * H * I
    proto = (torch.randn(nel, generator=torch.Generator().manual_seed(3)) * 0.02).to(dtype)
    blobs = {}
    for l in range(L):
        for e in range(E):
            b = torch.empty(nel, dtype=dtype, pin_memory=True)
            b.copy_(proto)
            b[:4096] += 0.001 * (l * E + e)
            blobs[(l, e)] = b
    pin_s = time.perf_counter() - t0
    # ---- trace: gates with a bias column, hidden states correlated over steps and layers
    g = torch.Generator(device="cpu").manual_seed(11)
    cconst = 4.0
    gates = []
    for l in range(L):
        w = torch.randn(E, H, generator=g) * 0.02
        perm = torch.randperm(E, generator=g)
        bias = (-args.skew * torch.log(torch.arange(1, E + 1).float()))[perm]
        w[:, H - 1] = bias / cconst
        gates.append(w)
    rho_s, rho_l = 0.9, 0.9
    xs = torch.empty(steps + warm, L, T, H, dtype=dtype).pin_memory()
    h = torch.randn(L, T, H, generator=g)
    for s_ in range(steps + warm):
        n = torch.randn(L, T, H, generator=g)
        for l in range(1, L):
            n[l] = rho_l * n[l - 1] + (1 - rho_l ** 2) ** 0.5 * n[l]
        h = rho_s * h + (1 - rho_s ** 2) ** 0.5 * n
        hs = h.clone()
        hs[..., H - 1] = cconst
        xs[s_] = hs.to(dtype)
    xp = (torch.randn(args.prefill, H, generator=g)).to(dtype) if args.prefill else None
    if xp is not None:
        xp[:, H - 1] = cconst

    def run(policy, lookahead, tag):
        eng = MoEEngine(num_layers=L, num_experts=E, hidden=H, inter=I, top_k=k, dtype=dtype,
                        max_tokens=max(16, args.prefill), device_memory_ratio=ratio, cache_policy=policy,
                        lookahead_prefetch=lookahead, max_inflight_prefetch=args.inflight,
                        h2d_chunk_bytes=args.chunk_mb << 20)
        for (l, e), b in blobs.items():
            eng._blobs[(l, e)] = b
            eng._ck(eng.lib.b2m_register_expert(eng._h, l, e, C.c_void_p(b.data_ptr()), b.numel() * 2))
        for l in range(L):
            eng.set_gate(l, gates[l].to(dtype))
        x_dev = torch.empty(L, T, H, dtype=dtype, device=dev)
        out_dev = torch.empty_like(x_dev)
        out_host = torch.empty(L, T, H, dtype=dtype).pin_memory()
        prefill_ms = None
        if xp is not None:
            xpd = xp.to(dev)
            op = torch.empty_like(xpd)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for l in range(L):
                eng.forward(l, xpd, out=op)
            torch.cuda.synchronize()
            prefill_ms = (time.perf_counter() - t0) * 1e3
            del xpd, op
            eng.clear_expert_cache_counts()          # what the reference's example does after prefill (interface_example.py:39)

        def step(i):
            x_dev.copy_(xs[i], non_blocking=True)
            for l in range(L):
                eng.forward(l, x_dev[l], out=out_dev[l])
            out_host.copy_(out_dev, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        for i in range(warm):
            step(i)
        s0 = eng.stats()
        times = []
        for i in range(steps):
            t0 = time.perf_counter()
            step(warm + i)
            times.append(time.perf_counter() - t0)
        s1 = eng.stats()
        d = {kk: s1[kk] - s0[kk] for kk in s1 if kk not in ("slots", "slot_bytes", "resident")}
        tot = sum(times)
        res = {"policy": tag, "slots": s1["slots"], "experts": L * E, "ms_per_step": tot / steps * 1e3,
               "p50_ms": sorted(times)[len(times) // 2] * 1e3, "tokens_per_s": T * steps / tot,
               "hit_rate": d["hits"] / max(1, d["dispatches"]), "dispatches_per_step": d["dispatches"] / steps,
               "misses_per_step": d["misses"] / steps, "h2d_gb_per_step": d["h2d_bytes"] / steps / 1e9,
               "h2d_gbs": d["h2d_bytes"] / tot / 1e9, "link_frac": d["h2d_bytes"] / tot / 1e9 / h2d_peak,
               "prefetch_issued_per_step": d["prefetch_issued"] / steps, "prefetch_useful_per_step": d["prefetch_useful"] / steps,
               "evictions_per_step": d["evictions"] / steps, "host_syncs_per_step": d["host_syncs"] / steps,
               "kernel_launches_per_step": d["kernel_launches"] / steps, "prefill_ms": prefill_ms,
               "out_checksum": float(out_host.float().abs().sum())}
        eng.prefetch_drain()
        eng.close()
        del eng
        torch.cuda.empty_cache()
        return res

    sampler = ClockSampler(0)
    sampler.start()
    ref = run(L_.CACHE_REFERENCE, 0, "reference (on-demand, evict min incache_visit_count; prefetch off)")
    ours = run(L_.CACHE_ACTIVATION_AWARE, 1, "activation-aware cache + router-logit look-ahead prefetch into idle link time")
    extra = {}
    if args.ablate:
        extra["activation_aware_no_prefetch"] = run(L_.CACHE_ACTIVATION_AWARE, 0, "activation-aware cache, prefetch off")
        extra["activation_aware_prefetch_always"] = run(L_.CACHE_ACTIVATION_AWARE, 2, "activation-aware cache + unconditional look-ahead prefetch")
    clocks = sampler.stop()
    line = {
        "metric": METRIC, "value": ours["tokens_per_s"], "unit": "tokens/s", "n_gpus": 1, "steps": steps, "warmup": warm,
        "ms_per_step": ours["ms_per_step"], "p50_token_latency_ms": ours["p50_ms"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"Mixtral-8x7B MoE dispatch path, forced offload: device_memory_ratio={ratio} -> {ours['slots']} of "
                               f"{L * E} experts HBM resident, the rest staged from pinned host DRAM on demand / ahead; decode "
                               f"batch {BATCH}, {L} layers, Zipf-{args.skew} routing, hidden states AR(1) 0.9 over steps and layers, "
                               f"after a T={args.prefill} prefill", "global_batch": BATCH, "layers": L, "parallelism": "single GPU",
                   "l2": "inputs larger than L2 (every miss streams a 352 MB expert)", "numerics": "reference rounding chain",
                   "timed_region": "host API per layer (MoEEngine.forward), inputs from pinned host memory, outputs back, host synchronised"},
        "roofline": {"bound": "h2d link", "kernel": "cudaMemcpyAsync H2D (expert staging)", "achieved": ours["h2d_gbs"],
                     "peak": h2d_peak, "unit": "GB/s", "frac": ours["link_frac"], "peak_source": "measured in this run (pinned 1 GiB copies)",
                     "algorithmic_bytes_per_step": ours["misses_per_step"] * 3 * H * I * 2, "traffic": None},
        "e2e": {"value": ours["tokens_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": L * T * H * 2 + int(ours["h2d_gb_per_step"] * 1e9),
                "d2h_bytes_per_step": L * T * H * 2},
        "gpu_launches": int(ours["kernel_launches_per_step"] * steps), "clocks": clocks,
        "ours": ours, "reference_policy": ref, "speedup_vs_reference_policy": ours["tokens_per_s"] / ref["tokens_per_s"],
        "same_outputs": abs(ours["out_checksum"] - ref["out_checksum"]) <= 1e-6 * abs(ref["out_checksum"]),
        "pin_seconds": pin_s, **extra,
    }
    print(json.dumps(line), flush=True)


def run_deepseek(args):
    """--config deepseek = BASELINE configs[3]: DeepSeek-V2-Lite (26 MoE layers, 64 routed experts top-6 + 2 shared,
    H=2048, moe I=1408), bf16 random-init, batch 16: decode T=16 tokens/layer/step (value, HBM roofline) and the prefill of
    16 x 4096 = 65536 tokens through all layers (tensor-core roofline), everything HBM resident (29.7 GB)."""
    from moe_infinity_b200 import MoEEngine, _lib as L_
    from moe_infinity_b200.engine import _view
    import ctypes as C
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    Hh, I, E, k, Lr = 2048, 1408, 64, 6, (args.layers or 26)
    Tp = args.prefill if args.prefill != 16384 else 65536
    dtype = torch.bfloat16
    eng = MoEEngine(num_layers=Lr, num_experts=E, hidden=Hh, inter=I, top_k=k, dtype=dtype, expert_type=L_.EXPERT_DEEPSEEK,
                    router=L_.ROUTER_DEEPSEEK_GREEDY, shared_inter=2 * I, max_tokens=max(Tp, 16), num_slots=Lr * E)
    for l in range(Lr):
        for e in range(E):
            eng.load_expert(l, e).normal_(0, 0.02)
        eng.set_gate(l, torch.randn(E, Hh, device=dev) * 0.05)
        p = C.c_void_p()
        eng._ck(eng.lib.b2m_shared_dev_ptr(eng._h, l, C.byref(p)))
        _view(p.value, (3 * Hh * 2 * I,), dtype, eng.device).normal_(0, 0.02)
        eng._ck(eng.lib.b2m_register_shared(eng._h, l, None, 0))
    peak, peak_src = load_peaks()
    tf_peak, tf_src = 1417.8, "fallback (no MEASURED_PEAKS.json)"
    if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")):
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            tf_peak = float(json.load(f).get("bf16_tflops_sustained", tf_peak))
        tf_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"

    def measure(T, iters, graph=True):
        x = torch.randn(Lr, T, Hh, device=dev).to(dtype)
        out = torch.empty_like(x)

        def step():
            for l in range(Lr):
                eng.forward(l, x[l], out=out[l])
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        l0 = eng.stats()["kernel_launches"]
        step()
        launches = eng.stats()["kernel_launches"] - l0
        counts = []
        for l in range(Lr):
            eng.route(l, x[l])
            counts.append(int((eng.ws("counts", T) > 0).sum()))
        run = step
        if graph:
            g = torch.cuda.CUDAGraph()
            s_ = torch.cuda.Stream()
            s_.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s_):
                step()
            torch.cuda.current_stream().wait_stream(s_)
            with torch.cuda.graph(g):
                step()
            run = g.replay
        for _ in range(2):
            run()
        torch.cuda.synchronize()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
        evs[0].record()
        for i in range(iters):
            run()
            evs[i + 1].record()
        torch.cuda.synchronize()
        ms = evs[0].elapsed_time(evs[-1]) / iters
        per = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(iters))
        bytes_step = sum(a * 3 * Hh * I * 2 for a in counts) + Lr * 3 * Hh * 2 * I * 2 + Lr * (2 * T * Hh * 2 + T * E * 4 + T * k * 8)
        flops = Lr * T * (k + 2) * 6 * Hh * I
        # e2e through the public API with host buffers
        xh, oh = x.cpu().pin_memory(), torch.empty_like(x).cpu().pin_memory()
        xin = torch.empty_like(x)

        def step_e2e():
            xin.copy_(xh, non_blocking=True)
            for l in range(Lr):
                eng.forward(l, xin[l], out=out[l])
            oh.copy_(out, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        step_e2e()
        t0 = time.perf_counter()
        n_e2e = max(2, iters // 2)
        for _ in range(n_e2e):
            step_e2e()
        e2e_ms = (time.perf_counter() - t0) * 1e3 / n_e2e
        return {"T": T, "ms_per_step": ms, "p50_ms": per[len(per) // 2], "tokens_per_s": T / ms * 1e3,
                "avg_active_experts": sum(counts) / len(counts), "algorithmic_bytes": bytes_step, "hbm_gbs": bytes_step / ms / 1e6,
                "hbm_frac": bytes_step / ms / 1e6 / peak, "tflops": flops / ms / 1e9, "tensor_frac": flops / ms / 1e9 / tf_peak,
                "launches_per_step": launches, "e2e_ms_per_step": e2e_ms, "e2e_tokens_per_s": T / e2e_ms * 1e3,
                "h2d_bytes": xh.numel() * 2, "d2h_bytes": oh.numel() * 2}

    sampler = ClockSampler(0)
    sampler.start()
    dec = measure(16, args.steps)
    clocks = sampler.stop()
    pre = measure(Tp, 3, graph=False) if Tp > 0 else None
    line = {
        "metric": "decode tokens/sec + p50 per-token latency, DeepSeek-V2-Lite MoE dispatch path", "value": dec["tokens_per_s"],
        "unit": "tokens/s", "n_gpus": 1, "steps": args.steps, "warmup": 2, "ms_per_step": dec["ms_per_step"],
        "p50_token_latency_ms": dec["p50_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": f"DeepSeek-V2-Lite MoE dispatch path: {Lr} MoE layers x 64 routed experts top-6 + 2 shared, H=2048 "
                               f"I=1408, bf16 random-init, batch 16: decode T=16 tokens/layer/step; all experts HBM resident",
                   "global_batch": 16, "layers": Lr, "parallelism": "single GPU",
                   "l2": "inputs larger than L2 (a step streams %.1f GB of expert weights)" % (dec["algorithmic_bytes"] / 1e9),
                   "numerics": "reference rounding chain", "timed_region": "CUDA graph replay of the step"},
        "roofline": {"bound": "hbm", "kernel": "whole step (grouped gate/up + down GEMMs dominate)", "achieved": dec["hbm_gbs"], "peak": peak,
                     "unit": "GB/s", "frac": dec["hbm_frac"], "peak_source": peak_src, "traffic": None,
                     "algorithmic_bytes_per_step": dec["algorithmic_bytes"]},
        "e2e": {"value": dec["e2e_tokens_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": dec["h2d_bytes"],
                "d2h_bytes_per_step": dec["d2h_bytes"], "ms_per_step": dec["e2e_ms_per_step"]},
        "gpu_launches": int(dec["launches_per_step"] * args.steps), "clocks": clocks, "decode": dec,
        "prefill": None if pre is None else dict(pre, roofline={"bound": "tensor", "achieved": pre["tflops"], "peak": tf_peak,
                                                               "unit": "TFLOP/s", "frac": pre["tensor_frac"],
                                                               "peak_source": tf_src}),
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="mixtral", choices=["mixtral", "offload", "deepseek"],
                    help="mixtral = BASELINE configs[1] (headline, default); offload = configs[2] (device_memory_ratio 0.25); "
                         "deepseek = configs[3] (DeepSeek-V2-Lite, batch 16)")
    ap.add_argument("--ratio", type=float, default=0.25, help="offload: device_memory_ratio")
    ap.add_argument("--skew", type=float, default=1.0, help="offload: Zipf exponent of the per-layer expert popularity")
    ap.add_argument("--prefill", type=int, default=16384, help="offload: tokens of the prefill that precedes the decode steps (0 = none)")
    ap.add_argument("--inflight", type=int, default=2, help="offload: concurrent prefetch copies")
    ap.add_argument("--chunk-mb", type=int, default=0, help="offload: H2D copy granularity (0 = whole expert)")
    ap.add_argument("--ablate", action="store_true", help="offload: also run the two half-way configurations")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layers", type=int, default=0, help="debug: fewer layers (invalid as a bench value)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (float32; single-GPU mixtral path)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "mixtral" or args.gpus != 1):
        ap.error("--dump-outputs covers the single-GPU mixtral path (--config mixtral --gpus 1 --impl ours)")
    if args.impl == "reference":
        return run_reference(args)
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: bench.py measures the CUDA path only"}))
        sys.exit(2)
    if args.config == "offload":
        return run_offload(args)
    if args.config == "deepseek":
        return run_deepseek(args)
    run_ours(args)


if __name__ == "__main__":
    main()
