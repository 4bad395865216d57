import numpy as np


def grid(n, d, seed):
    """Quantised-grid data (coordinates j/64, |j| <= 8): products and partial sums are exact in fp32 and bf16, so
    scores are identical under ANY summation order and ties are abundant (SURVEY.md §7 'Hard parts')."""
    rng = np.random.default_rng(seed)
    return (rng.integers(-8, 9, size=(n, d)).astype(np.float32) / 64).astype(np.float32)


def gauss(n, d, seed, normalize=True):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, d), dtype=np.float32)
    if normalize:
        x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


class NumpyVS:
    """Test double of the VS plugin surface (lotus/vector_store/vs.py) backed by the oracle: lets the pandas
    operators be exercised on CPU. It lives in tests/ only — the product has no CPU path."""

    supports_ids_search = True

    def __init__(self, metric=0):
        self.metric = metric
        self.index_dir = None
        self.dirs = {}
        self.x = None

    def index(self, docs, embeddings, index_dir, **kw):
        self.dirs[index_dir] = np.asarray(embeddings, dtype=np.float32)
        self.index_dir = index_dir
        self.x = self.dirs[index_dir]

    def load_index(self, index_dir):
        if index_dir not in self.dirs:
            raise ValueError(f"Index directory {index_dir} not found")
        self.index_dir = index_dir
        self.x = self.dirs[index_dir]

    def get_vectors_from_index(self, index_dir, ids):
        return self.dirs[index_dir][np.asarray(list(ids), dtype=np.int64)]

    def __call__(self, query_vectors, K, ids=None, **kw):
        import oracle
        from lotus_b200.types import RMOutput
        if self.x is None:
            raise ValueError("Index not loaded")
        q = np.asarray(query_vectors, dtype=np.float32)
        if ids is None:
            D, I = oracle.knn(self.x, q, K, self.metric)
        else:
            D, I = oracle.knn_subset(self.x, q, K, np.asarray(list(ids), dtype=np.int64), self.metric)
        return RMOutput(distances=D, indices=I)

    # extension methods the re-registered accessors use (oracle-backed, tests only)
    def threshold_pairs(self, threshold):
        import oracle
        pi, pj, _ = oracle.threshold_pairs(self.x, float(threshold))
        return pi, pj

    def kmeans(self, ids, ncentroids, niter=20, seed=1234, full_lloyd=False):
        import oracle
        return oracle.kmeans(self.x[np.asarray(ids, dtype=np.int64)], ncentroids, niter=niter, seed=seed, full_lloyd=full_lloyd)


def frame_from_json(j):
    import pandas as pd
    return pd.DataFrame(j["data"], columns=j["columns"], index=j["index"])


def assert_frame_matches_json(df, j):
    """DataFrame equals a fixture produced by the reference's operator code (tests/golden/reference_ops.json)."""
    assert [str(c) for c in df.columns] == j["columns"]
    assert [int(i) for i in df.index] == j["index"]
    got = df.to_numpy().tolist()
    assert len(got) == len(j["data"])
    for r_got, r_want in zip(got, j["data"]):
        for a, b in zip(r_got, r_want):
            if isinstance(b, float):
                assert np.float32(a) == np.float32(b), (a, b)
            else:
                assert a == b, (a, b)


def replay_reference_vs_calls(vs, root):
    """Makes on `vs` every vector-store call the reference's own operators (sem_index, sem_sim_join, sem_search, sem_dedup,
    sem_cluster_by) made on its FaissVS when tests/golden/reference_ops.json was generated — same arguments, same argument
    types — and asserts FaissVS's answers (tests/golden/reference_vs_calls.*, make_reference_golden.py). Those operators
    build their frames from nothing else, so a store that passes answers them as FaissVS did. One documented divergence:
    past the last candidate (K > rows searched) FaissVS wraps the -1 pad to the last id (faiss_vs.py:71-72); `vs` must
    pad with -1. Returns the number of calls replayed."""
    import json
    import os

    import pandas as pd
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    with open(os.path.join(golden, "reference_vs_calls.json")) as f:
        calls = json.load(f)["calls"]
    arrays = np.load(os.path.join(golden, "reference_vs_calls.npz"))
    rows = {}
    for n, c in enumerate(calls):
        where = (n, c["op"])
        if c["op"] == "index":
            emb = arrays[c["embeddings"]]
            vs.index(pd.Series(c["docs"]), emb, os.path.join(root, c["dir"]))
            rows[c["dir"]] = len(emb)
            assert vs.index_dir == os.path.join(root, c["dir"]), where
        elif c["op"] == "load_index":
            vs.load_index(os.path.join(root, c["dir"]))
            assert vs.index_dir == os.path.join(root, c["dir"]), where
        elif c["op"] == "get_vectors_from_index":
            ids = pd.Index(c["ids"]) if c["ids_type"] == "pandas.Index" else c["ids"]
            got = np.asarray(vs.get_vectors_from_index(os.path.join(root, c["dir"]), ids))
            assert np.array_equal(bits(got), bits(arrays[c["out"]])), where
        else:
            out = vs(arrays[c["query"]], c["K"], ids=c["ids"])
            D, I = np.asarray(out.distances), np.asarray(out.indices)
            want_D, want_I = arrays[c["distances"]], arrays[c["indices"]]
            assert D.shape == want_D.shape and I.shape == want_I.shape, where
            m = min(c["K"], rows[os.path.relpath(vs.index_dir, root)] if c["ids"] is None else len(c["ids"]))
            assert np.array_equal(I[:, :m], want_I[:, :m]), where
            assert np.array_equal(bits(D[:, :m]), bits(want_D[:, :m])), where
            assert (I[:, m:] == -1).all(), where
    return len(calls)


def _nv():
    from lotus_b200 import _native
    return _native


import oracle  # noqa: E402  (test infrastructure: the fake index below is the oracle behind B200VS's native calls)


class FakeIndex:
    """Stands in for _nv().Index: same constructor, attributes and methods, computed by the oracle."""
    live = 0

    def __init__(self, x, dtype, metric=0, device=0, on_device_ptr=None, n=None, d=None):
        assert on_device_ptr is None
        x = np.ascontiguousarray(x)
        assert x.dtype == (np.float32 if dtype == _nv().F32 else np.uint16) and x.ndim == 2
        self.raw, self.dtype, self.metric, self.device = x, dtype, metric, device
        self.vals = x if dtype == _nv().F32 else _nv().bf16_bits_to_f32(x)
        self.n, self.d = x.shape
        self.closed = False
        self.calls = []
        FakeIndex.live += 1

    def close(self):
        if not self.closed:
            self.closed = True
            FakeIndex.live -= 1

    def search(self, q, k, q_dtype=0, ids=None):
        assert not self.closed
        self.calls.append((q.dtype, q_dtype, None if ids is None else len(ids)))
        if k > 2048:
            raise _nv().NativeError(_nv().ERANGE, f"k={k} is not supported")
        qv = q if q_dtype == _nv().F32 else _nv().bf16_bits_to_f32(q)
        if ids is None:
            return oracle.knn(self.vals, qv, k, self.metric)
        if len(ids) and (ids.min() < 0 or ids.max() >= self.n):
            raise _nv().NativeError(_nv().ERANGE, f"ids contains a position outside [0, {self.n})")
        return oracle.knn_subset(self.vals, qv, k, ids, self.metric)

    def gather(self, ids):
        return self.raw[np.asarray(ids, dtype=np.int64)]

    def threshold_pairs(self, thr, cap=1 << 24, part=0, nparts=1):
        import oracle
        pi, pj, _ = oracle.threshold_pairs(self.vals, float(thr))
        return pi, pj

    def kmeans(self, k, niter=20, seed=1234, ids=None, full_lloyd=False):
        import oracle
        x = self.vals if ids is None else self.vals[np.asarray(ids, dtype=np.int64)]
        return oracle.kmeans(np.ascontiguousarray(x), k, niter=niter, full_lloyd=full_lloyd)

