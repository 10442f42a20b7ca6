"""TEST INFRASTRUCTURE — seeded inputs for the Megatron index builders (`helpers`: build_sample_idx, build_mapping,
build_blocks_mapping, build_blending_indices). `run_cases(helpers_module)` runs them against ANY implementation with the
reference's call signatures: oracle/make_golden_index_builders.py feeds it the reference's own C++ compiled into oracle/_ref/
(-> tests/golden/index_builders.npz), tests/test_index_builders_cpu.py feeds it the fsb200 compat module and compares.
`random_cases` does the same on randomised inputs; its reference outputs are kept as digests
(oracle/make_golden_reference_runs.py -> tests/golden/index_builders_random.json)."""
import hashlib

import numpy as np


def corpus(rs, n_docs, max_sent=9, max_len=90, p_empty=0.05, p_long=0.03):
    """docs[n_docs + 1] (first sentence of each document), sizes[sentence]. Includes empty and one-sentence documents and a few
    sentences longer than 512 tokens (documents holding one are skipped by the builders)."""
    n_sent = rs.randint(0, max_sent + 1, size=n_docs)
    n_sent[rs.rand(n_docs) < p_empty] = 0
    docs = np.concatenate([[0], np.cumsum(n_sent)]).astype(np.int64)
    sizes = rs.randint(1, max_len + 1, size=int(docs[-1])).astype(np.int32)
    sizes[rs.rand(sizes.shape[0]) < p_long] = 513 + rs.randint(0, 100)
    return docs, sizes


def run_cases(H):
    out = {}
    rs = np.random.RandomState(2024)
    # ---- build_sample_idx: documents of 0..40 tokens (zero-length ones included), several epochs of a shuffled order
    for i, (n_docs, seq, epochs) in enumerate(((50, 16, 1), (200, 64, 3), (7, 5, 2), (1000, 2048, 2), (3, 2, 4))):
        sizes = rs.randint(0, 41, size=n_docs).astype(np.int32)
        sizes[rs.randint(0, n_docs)] += seq + 3           # at least one document longer than a sample
        order = np.concatenate([rs.permutation(n_docs) for _ in range(epochs)]).astype(np.int32)
        tokens_per_epoch = int(sizes.sum())
        out[f"sample_idx_{i}"] = np.asarray(H.build_sample_idx(sizes, order, seq, epochs, tokens_per_epoch))
    # ---- build_mapping
    k = 0
    for n_docs in (1, 40, 300):
        docs, sizes = corpus(rs, n_docs)
        for (epochs, max_samples, max_len, p_short, seed, min_sent) in (
                (1, 10 ** 9, 128, 0.0, 1234, 2), (3, 10 ** 9, 128, 0.1, 7, 2), (2, 25, 64, 0.5, 99, 1),
                (4, 10 ** 9, 512, 1.0, 3, 2), (2, 10 ** 9, 32, 0.25, 2 ** 31 - 2, 3)):
            out[f"mapping_{k}"] = np.asarray(H.build_mapping(docs, sizes, epochs, max_samples, max_len, p_short, seed, False,
                                                             min_sent))
            k += 1
    # ---- build_blocks_mapping
    k = 0
    for n_docs in (1, 40, 300):
        docs, sizes = corpus(rs, n_docs)
        titles = rs.randint(0, 20, size=n_docs).astype(np.int32)
        for (epochs, max_samples, max_len, seed, one_sent) in ((1, 10 ** 9, 128, 1234, False), (3, 10 ** 9, 64, 5, True),
                                                               (2, 30, 256, 77, False), (2, 10 ** 9, 40, 11, True)):
            out[f"blocks_{k}"] = np.asarray(H.build_blocks_mapping(docs, sizes, titles, epochs, max_samples, max_len, seed,
                                                                   False, one_sent))
            k += 1
    # ---- build_blending_indices
    for i, (w, size) in enumerate((([1.0], 10), ([0.5, 0.5], 33), ([0.7, 0.2, 0.1], 1000), ([0.25] * 4, 101),
                                   (list(np.random.RandomState(5).dirichlet(np.ones(9))), 5000), ([0.9, 0.1], 0))):
        di = np.zeros(size, dtype=np.uint8)
        ds = np.zeros(size, dtype=np.int64)
        H.build_blending_indices(di, ds, np.asarray(w, dtype=np.float64), len(w), size, False)
        out[f"blend_index_{i}"], out[f"blend_sample_{i}"] = di, ds
    return out


def digest(a):
    """SHA-256 of an array's dtype, shape and bytes: exact equality at a fraction of the array's size."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def random_cases(H, trials=40):
    """Randomised corpora and arguments (seed 31337), every builder per trial: `{trial}_mapping`, `_blocks`, `_sample_idx`,
    `_blend_index`, `_blend_sample`."""
    out = {}
    rs = np.random.RandomState(31337)
    for trial in range(trials):
        n_docs = int(rs.randint(1, 400))
        docs, sizes = corpus(rs, n_docs, max_sent=int(rs.randint(1, 15)), max_len=int(rs.randint(2, 200)),
                             p_empty=rs.rand() * 0.3, p_long=rs.rand() * 0.05)
        titles = rs.randint(0, 30, size=n_docs).astype(np.int32)
        epochs, seed = int(rs.randint(1, 5)), int(rs.randint(1, 2 ** 31 - 1))
        cap = int(rs.choice([10 ** 9, rs.randint(1, 200)]))
        max_len = int(rs.randint(8, 600))
        p_short = float(rs.choice([0.0, 0.1, 0.33, 1.0]))
        min_sent = int(rs.randint(1, 4))
        one = bool(rs.randint(0, 2))
        out[f"{trial}_mapping"] = np.asarray(H.build_mapping(docs, sizes, epochs, cap, max_len, p_short, seed, False, min_sent))
        out[f"{trial}_blocks"] = np.asarray(H.build_blocks_mapping(docs, sizes, titles, epochs, cap, max_len, seed, False, one))
        tok = rs.randint(0, 60, size=n_docs).astype(np.int32)
        seq = int(rs.randint(2, 100))
        tok[rs.randint(0, n_docs)] += seq + 1
        order = np.concatenate([rs.permutation(n_docs) for _ in range(epochs)]).astype(np.int32)
        out[f"{trial}_sample_idx"] = np.asarray(H.build_sample_idx(tok, order, seq, epochs, int(tok.sum())))
        nd = int(rs.randint(1, 12))
        w = rs.dirichlet(np.ones(nd))
        size = int(rs.randint(0, 3000))
        a, b = np.zeros(size, np.uint8), np.zeros(size, np.int64)
        H.build_blending_indices(a, b, w, nd, size, False)
        out[f"{trial}_blend_index"], out[f"{trial}_blend_sample"] = a, b
    return out
