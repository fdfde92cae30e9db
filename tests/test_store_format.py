"""CPU: the reference's on-disk tensor store format (moe_infinity_b200/store.py) against the reference's own code.

  * golden: tests/golden/archer_index_ref.bin was written by `ArcherTensorIndex::Serialize`
    (core/aio/archer_tensor_index.cpp:105-113 compiled as-is, tests/golden/make_store_golden.py) -- always checked;
  * round trip on random tensor sets: our writer -> the reference's `Deserialize`, the reference's `Serialize` -> our
    parser (what the reference code read and wrote is recorded in tests/golden/reference_results.pt by
    tests/golden/make_reference_golden.py; our writer must still produce the bytes it read);
  * the data files: 4096-byte aligned offsets (kAioAlignment), whole aligned blocks on disk, StoreTensor's rules for
    known ids, reload, expert blobs, and the opt-in persistent mode of compat.prefetch_handle.
Bit-exact: it is a byte format."""
from __future__ import annotations

import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))

from make_store_golden import STORE_GOLDEN_ENTRIES  # noqa: E402
from reference_cases import STORE_SEEDS, random_tensors  # noqa: E402
from moe_infinity_b200.store import ALIGN, ArcherTensorStore, TensorMeta, parse_index, serialize_index  # noqa: E402

REF = torch.load(os.path.join(HERE, "golden", "reference_results.pt"), weights_only=False)["store"]
_SCALAR = {torch.uint8: 0, torch.int64: 4, torch.float16: 5, torch.float32: 6, torch.bfloat16: 15, torch.float8_e4m3fn: 24}


def test_parser_reads_the_reference_writers_file():
    with open(os.path.join(HERE, "golden", "archer_index_ref.bin"), "rb") as f:
        data = f.read()
    idx = parse_index(data)
    assert sorted(idx) == sorted(e[0] for e in STORE_GOLDEN_ENTRIES)
    for tid, file_id, offset, shape, dt in STORE_GOLDEN_ENTRIES:
        m = idx[tid]
        numel = 1
        for d in shape:
            numel *= d
        assert (m.file_id, m.offset, m.shape, m.scalar_type) == (file_id, offset, shape, _SCALAR[dt])
        assert m.size == numel * torch.empty(0, dtype=dt).element_size()
        assert (m.pinned, m.requires_grad, m.device_type, m.device_index, m.layout) == (False, False, 0, -1, 0)
        assert m.dtype == dt
    # our writer emits the same bytes per entry (entry ORDER is the reference's unordered_map order, so compare as sets)
    again = parse_index(serialize_index(idx))
    assert again == idx and len(serialize_index(idx)) == len(data)
    for bad in (data[:3], data[:40], data[:-1]):
        with pytest.raises(ValueError):
            parse_index(bad)


def test_round_trip_with_the_compiled_reference_index_code(tmp_path):
    for seed in STORE_SEEDS:
        ref = REF[seed]
        tensors = random_tensors(seed, 25)
        d = tmp_path / f"s{seed}"
        store = ArcherTensorStore(str(d))
        for tid, t in tensors.items():
            store.store_tensor(tid, t, flush=False)
        store.flush()
        # ours -> reference reader: the file is the one the reader read, and what it read is what we meant
        with open(store.index_path, "rb") as f:
            assert f.read() == ref["our_index"]
        got = ref["ref_deserialize"]
        assert sorted(got) == sorted(tensors)
        for tid, t in tensors.items():
            m = store.index[tid]
            assert got[tid] == (m.file_id, m.offset, t.numel() * t.element_size(), list(t.shape), m.scalar_type, 0, -1, 0,
                                False, False)
        # reference writer -> ours (same metas, built by the reference from the tensors themselves)
        assert parse_index(ref["ref_index"]) == store.index


def test_data_file_layout_and_store_rules(tmp_path):
    d = str(tmp_path / "store")
    s = ArcherTensorStore(d)
    assert not s.is_initialized() and len(s) == 0 and os.path.isdir(d)
    a = torch.randn(100, 33).to(torch.bfloat16)          # 6600 B -> 2 blocks
    b = torch.randn(5)                                   # 20 B
    c = torch.arange(1025, dtype=torch.int64)            # 8200 B -> 3 blocks
    for tid, t in ((3, a), (1, b), (2, c)):
        s.store_tensor(tid, t)
    assert [s.index[i].offset for i in (3, 1, 2)] == [0, 2 * ALIGN, 3 * ALIGN]           # archer_tensor_handle.cpp:64-78
    assert all(s.index[i].file_id == 0 for i in (1, 2, 3)) and s.aligned_size(2) == 3 * ALIGN
    assert os.path.getsize(s.param_path(0)) == 6 * ALIGN                                  # whole aligned blocks
    raw = open(s.param_path(0), "rb").read()
    assert raw[:6600] == a.view(torch.uint8).numpy().tobytes() and raw[2 * ALIGN:2 * ALIGN + 20] == b.numpy().tobytes()
    # known id: same size -> rewritten in place, nothing moves; other size -> refused (the reference aborts, :70-74)
    a2 = torch.randn(100, 33).to(torch.bfloat16)
    s.store_tensor(3, a2)
    assert s.index[3].offset == 0 and torch.equal(s.read_tensor(3), a2) and torch.equal(s.read_tensor(1), b)
    with pytest.raises(ValueError, match="size mismatch"):
        s.store_tensor(3, torch.zeros(7))
    # reload: initialised, same contents, new ids are appended behind the last stored block
    s2 = ArcherTensorStore(d + "/")
    assert s2.is_initialized() and s2.index == s.index and 2 in s2 and 99 not in s2
    assert torch.equal(s2.read_tensor(2), c) and s2.read_tensor(2).dtype == torch.int64
    s2.store_tensor(9, torch.ones(3, dtype=torch.float16))
    assert s2.index[9].offset == 6 * ALIGN and torch.equal(s2.read_tensor(3), a2)
    # expert blob = tensors of an expert concatenated in id order, no padding
    blob = s2.read_expert_blob([3, 1, 9])
    want = a2.view(torch.uint8).reshape(-1).tolist() + b.view(torch.uint8).tolist() + torch.ones(3, dtype=torch.float16).view(torch.uint8).tolist()
    assert blob.dtype == torch.uint8 and blob.tolist() == want
    with pytest.raises(ValueError):
        s2.read_into(2, torch.empty(10, dtype=torch.uint8))
    # a truncated data file is an error, not garbage
    with open(s2.param_path(0), "r+b") as f:
        f.truncate(ALIGN)
    with pytest.raises(IOError):
        s2.read_tensor(2)
    with pytest.raises(ValueError):
        ArcherTensorStore(s2.index_path)               # prefix exists and is not a directory (:32-34)


def test_compat_handle_persistent_mode(tmp_path):
    """model_offload.py:346-399: offload every checkpoint tensor once, later runs find `is_tensor_index_initialized()`."""
    from moe_infinity_b200 import compat
    d = str(tmp_path / "offload")
    w = {i: torch.randn(16, 8, generator=torch.Generator().manual_seed(i)).to(torch.bfloat16) for i in range(6)}
    h = compat.prefetch_handle(d, 0.5, persistent=True)
    assert not h.is_tensor_index_initialized()
    for i, t in w.items():
        assert not h.is_tensor_offloaded(i)
        h.offload(t, i)
        assert h.is_tensor_offloaded(i)
    h.flush()
    h2 = compat.prefetch_handle(d, 0.5, persistent=True)
    assert h2.is_tensor_index_initialized() and all(h2.is_tensor_offloaded(i) for i in w) and not h2.is_tensor_offloaded(77)
    assert all(torch.equal(h2._tensors[i], w[i]) for i in w)        # read back from disk on first use
    # the default handle never touches the disk
    h3 = compat.prefetch_handle(str(tmp_path / "never_created"), 0.5)
    h3.offload(w[0], 0)
    assert h3.is_tensor_offloaded(0) and not h3.is_tensor_index_initialized() and not os.path.exists(tmp_path / "never_created")
