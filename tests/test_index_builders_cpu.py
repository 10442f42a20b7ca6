"""Megatron index builders (SURVEY §8f rank 3: `helpers.cpp`) — fsb200's C-ABI implementation (`fsb_index_*`, host code inside
libfsb200.so, reached through compat `fengshen.data.megatron_dataloader.helpers`) against
  (1) golden vectors produced by the REFERENCE's own C++ (tests/golden/index_builders.npz, oracle/make_golden_index_builders.py),
  (2) digests of the reference's own C++ outputs on additional randomised inputs (tests/golden/index_builders_random.json,
      oracle/make_golden_reference_runs.py),
  (3) size-independent properties at a size the golden file does not hold (10 M tokens).
Integer work: the bar is exact equality, including the pseudo-random shuffles."""
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
for p in ("fengshen-lm_b200", os.path.join("fengshen-lm_b200", "compat")):
    sys.path.insert(0, os.path.join(ROOT, p))

import index_builder_cases as C  # noqa: E402


@pytest.fixture(scope="module")
def H():
    from fengshen.data.megatron_dataloader import helpers
    assert os.path.join("fengshen-lm_b200", "compat") in helpers.__file__
    return helpers


def test_matches_reference_golden_vectors(H):
    golden = np.load(os.path.join(ROOT, "tests", "golden", "index_builders.npz"))
    ours = C.run_cases(H)
    assert set(ours) == set(golden.files) and len(ours) == 44
    for k in golden.files:
        assert ours[k].dtype == golden[k].dtype and ours[k].shape == golden[k].shape, k
        assert np.array_equal(ours[k], golden[k]), k
    # not vacuous: mappings have rows, the short-sequence draw and the sample cap are exercised
    assert golden["mapping_6"].shape[0] > 100 and (golden["mapping_6"][:, 2] < 128).any()
    assert golden["mapping_7"].shape[0] <= 25 + 40 * 9


def test_matches_reference_on_random_inputs(H):
    """40 randomised corpora, every builder: equal to the reference's own C++ on the same inputs, recorded as digests in
    tests/golden/index_builders_random.json (oracle/make_golden_reference_runs.py)."""
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "index_builders_random.json")))
    ours = C.random_cases(H)
    assert len(ours) == 200
    for k, v in ours.items():
        assert C.digest(v) == golden[k], k


def test_sample_idx_properties_at_scale(H):
    """10 M tokens, seq 2048 (the C4 sequence length): every row addresses flattened position k * seq_length."""
    rs = np.random.RandomState(1)
    sizes = rs.randint(0, 3000, size=6700).astype(np.int32)
    epochs, seq = 2, 2048
    order = np.concatenate([rs.permutation(sizes.shape[0]) for _ in range(epochs)]).astype(np.int32)
    tokens = int(sizes.sum())
    idx = H.build_sample_idx(sizes, order, seq, epochs, tokens)
    n = (epochs * tokens - 1) // seq
    assert idx.shape == (n + 1, 2) and idx.dtype == np.int32 and n > 9000
    begin = np.concatenate([[0], np.cumsum(sizes[order].astype(np.int64))])
    pos = begin[idx[:, 0]] + idx[:, 1]
    assert np.array_equal(pos, np.arange(n + 1, dtype=np.int64) * seq)
    assert (idx[1:, 1] < sizes[order][idx[1:, 0]]).all() and (idx[:, 1] >= 0).all()
    assert (np.diff(idx[:, 0]) >= 0).all()


def test_mapping_properties_and_row_count_protocol(H):
    rs = np.random.RandomState(2)
    docs, sizes = C.corpus(rs, 5000)
    m = H.build_mapping(docs, sizes, 2, 10 ** 9, 512, 0.1, 1234, False, 2)
    assert m.dtype == np.uint32 and m.shape[1] == 3 and m.shape[0] > 5000
    first, end, target = m[:, 0].astype(np.int64), m[:, 1].astype(np.int64), m[:, 2]
    assert (end > first).all() and (target >= 2).all() and (target <= 512).all() and (target < 512).any()
    doc_of = np.searchsorted(docs, first, side="right") - 1
    assert (end <= docs[doc_of + 1]).all()                                   # a span never crosses a document
    assert not np.array_equal(first, np.sort(first))                         # shuffled
    # two epochs without a cap: every span appears... spans differ per epoch (targets are re-drawn), sentences covered twice
    covered = np.zeros(sizes.shape[0], dtype=np.int64)
    for a, b in zip(first, end):
        covered[a:b] += 1
    ok_docs = np.array([docs[d + 1] - docs[d] >= 2 and not (sizes[docs[d]:docs[d + 1]] > 512).any() for d in range(5000)])
    for d in np.nonzero(ok_docs)[0][:200]:
        assert (covered[docs[d]:docs[d + 1]] == 2).all()
    for d in np.nonzero(~ok_docs)[0][:200]:
        assert (covered[docs[d]:docs[d + 1]] == 0).all()
    # C-ABI protocol: wrong capacity is an error, not a silent truncation
    import ctypes
    from fsb200 import lib as L
    out = np.zeros((3, 3), dtype=np.uint32)
    fn = L.load().fsb_index_build_mapping
    rc = fn(ctypes.c_void_p(docs.ctypes.data), docs.shape[0] - 1, ctypes.c_void_p(sizes.ctypes.data), 2, 10 ** 9, 512, 0.1, 1234, 2,
            L.U32, ctypes.c_void_p(out.ctypes.data), 3)
    assert rc == -1 and "rows" in L.last_error()
    with pytest.raises(ValueError):
        H.build_sample_idx(sizes, np.zeros(4, np.int32), 1, 1, 100)


def test_blending_follows_weights(H):
    w = np.array([0.6, 0.3, 0.1])
    n = 100000
    di, ds = np.zeros(n, np.uint8), np.zeros(n, np.int64)
    H.build_blending_indices(di, ds, w, 3, n, False)
    counts = np.bincount(di, minlength=3)
    assert np.abs(counts / n - w).max() < 1e-4
    for d in range(3):
        assert np.array_equal(ds[di == d], np.arange(counts[d]))             # each dataset's samples are consumed in order
    with pytest.raises(TypeError):
        H.build_blending_indices(np.zeros(4, np.int32), ds, w, 3, 4, False)


def test_blendable_dataset_and_the_unmodified_reference_class_on_our_helpers(H):
    """The caller of build_blending_indices; its schedule equals the one the reference's BlendableDataset class builds on the
    reference's own helpers (tests/golden/index_builders_random.json)."""
    from fengshen.data.megatron_dataloader.blendable_dataset import BlendableDataset
    parts = [[("a", i) for i in range(70)], [("b", i) for i in range(20)], [("c", i) for i in range(10)]]
    ds = BlendableDataset(parts, [7, 2, 1])
    assert len(ds) == 100
    items = [ds[i] for i in range(100)]
    for name, n in (("a", 70), ("b", 20), ("c", 10)):
        assert [v for k, v in items if k == name] == list(range(n))          # everything consumed exactly once, in order
    assert [k for k, _ in items[:10]].count("a") == 7
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "index_builders_random.json")))
    assert np.array_equal(ds.dataset_index, golden["blendable_dataset_index"])
    assert np.array_equal(ds.dataset_sample_index, golden["blendable_dataset_sample_index"])
