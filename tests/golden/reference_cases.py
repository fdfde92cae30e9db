"""Seeded inputs shared by tests/golden/make_reference_golden.py (which records the reference's answers to them) and the
tests that compare against those answers (test_oracle_expert_ref, test_memory_policy, test_store_format)."""
from __future__ import annotations

import numpy as np
import torch

# expert module: (H, I, rows) per random case, every expert type x dtype
SHAPES = [(32, 48, 1), (64, 40, 13), (72, 136, 4), (256, 512, 33)]
PREDICTOR_SEEDS = [0, 1, 2]
PRIORITY_LAYERS = [0, 2, 3, 5]
STORE_SEEDS = range(4)


def rand_case(et, dt, H, I, n, seed):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: (torch.randn(*s, generator=g) * 0.1).to(dt)  # noqa: E731
    if et == 0:
        ws = [r(I, H), r(H, I)]
    elif et == 4:
        ws = [r(I, H), r(H, I), r(I, H)]
    elif et in (1, 5):
        ws = [r(I, H), r(I, H), r(H, I)]
    else:
        ws = [r(I, H), r(I), r(H, I), r(H)]
    return ws, torch.randn(n, H, generator=g).to(dt)


def seed_of(et, di, i):
    return 1000 + 17 * et + 5 * di + i


def library(rng, n, L, E):
    lib = rng.integers(0, 6, size=(n, L, E)).astype(np.float32)
    lib[:, :, 0] += 1.0   # no all-zero rows
    return lib


def prefetch_inputs(L, E):
    rng = np.random.default_rng(3)
    matrix = rng.random((L, E)) * (rng.random((L, E)) > 0.3)
    tmap = {(l, e): 100 + l * E + e for l in range(L) for e in range(E)}
    return matrix, tmap


def priority_inputs(current_layer):
    L, E = 6, 4
    rng = np.random.default_rng(current_layer)
    dec = rng.integers(0, 4, size=(L, E)).astype(np.float64)
    dec[1] = 0                                           # an all-zero layer row
    freq = {(int(e), int(l)): float(rng.integers(0, 5)) for l in range(L) for e in range(E) if rng.random() < 0.6}
    return L, E, dec, freq


def random_tensors(seed, n):
    g = torch.Generator().manual_seed(seed)
    dts = [torch.bfloat16, torch.float16, torch.float32, torch.int64, torch.uint8, torch.bool, torch.float64]
    out = {}
    for i in range(n):
        dt = dts[int(torch.randint(0, len(dts), (1,), generator=g))]
        rank = int(torch.randint(0, 4, (1,), generator=g))
        shape = [int(torch.randint(1, 40, (1,), generator=g)) for _ in range(rank)]
        t = (torch.randn(shape, generator=g) * 10)
        t = (t > 0) if dt == torch.bool else t.to(dt)
        out[int(torch.randint(0, 2 ** 31, (1,), generator=g)) * 2 + (i % 2)] = t
    return out
