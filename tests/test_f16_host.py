"""fp16 stores on CPU: the faiss IxSQ (IndexScalarQuantizer, QT_fp16) file layout, and the host semantics of
B200VS(dtype="f16") and B200VS(factory_string="SQfp16") over an oracle-backed fake of the native index (the real library runs
the same class in tests/test_gpu_f16.py). The SQfp16 contract is faiss's, as FaissVS uses it (faiss_vs.py:13-77): rows stored
as fp16 RNE of the embeddings, fp32 queries scored exactly against them, the `vecs` pickle and get_vectors_from_index keep the
originals."""
import os
import pickle
import struct

import numpy as np
import pytest

import oracle
from helpers import FakeIndex, gauss, grid
from lotus_b200 import _native as nv
from lotus_b200 import faiss_io
from lotus_b200.vs import B200VS


class F16FakeIndex(FakeIndex):
    """FakeIndex that also takes F16 matrices and F16 queries (uint16 bit patterns, like BF16)."""

    def __init__(self, x, dtype, metric=0, device=0, on_device_ptr=None, n=None, d=None):
        if dtype != nv.F16:
            super().__init__(x, dtype, metric, device, on_device_ptr, n, d)
            return
        assert on_device_ptr is None
        x = np.ascontiguousarray(x)
        assert x.dtype == np.uint16 and x.ndim == 2
        self.raw, self.dtype, self.metric, self.device = x, dtype, metric, device
        self.vals = nv.f16_bits_to_f32(x)
        self.n, self.d = x.shape
        self.closed = False
        self.calls = []
        FakeIndex.live += 1

    def search(self, q, k, q_dtype=0, ids=None):
        if q_dtype != nv.F16:
            return super().search(q, k, q_dtype, ids)
        self.calls.append((q.dtype, q_dtype, None if ids is None else len(ids)))
        qv = nv.f16_bits_to_f32(q)
        if ids is None:
            return oracle.knn(self.vals, qv, k, self.metric)
        return oracle.knn_subset(self.vals, qv, k, ids, self.metric)


@pytest.fixture
def fake_native(monkeypatch):
    FakeIndex.live = 0
    monkeypatch.setattr(nv, "Index", F16FakeIndex)
    monkeypatch.setattr(nv, "require_device", lambda: None)
    yield


def f16(x):
    return np.asarray(x, dtype=np.float32).astype(np.float16).astype(np.float32)


# ---- IxSQ layout ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", [faiss_io.METRIC_INNER_PRODUCT, faiss_io.METRIC_L2])
def test_ixsq_writer_matches_the_hand_assembled_layout(tmp_path, metric):
    x = np.array([[1.0, -2.5, 0.1], [65504.0, 1e-7, -0.0]], dtype=np.float32)
    n, d = x.shape
    want = (b"IxSQ" + struct.pack("<i", d) + struct.pack("<q", n) + struct.pack("<qq", 1 << 20, 1 << 20) + b"\x01"
            + struct.pack("<i", metric)
            + struct.pack("<i", 4) + struct.pack("<i", 0) + struct.pack("<f", 0.0)    # qtype QT_fp16, rangestat, rangestat_arg
            + struct.pack("<Q", d) + struct.pack("<Q", 2 * d)                          # d, code_size
            + struct.pack("<Q", 0)                                                     # trained: empty vector
            + struct.pack("<Q", n * 2 * d) + x.astype("<f2").tobytes())                # codes
    p = str(tmp_path / "index")
    faiss_io.write_sq_fp16_index(p, x.astype(np.float16), metric)
    assert open(p, "rb").read() == want
    y, m, kind = faiss_io.read_index(p)
    assert kind == faiss_io.SQFP16 and m == metric and y.dtype == np.float16
    assert np.array_equal(y.view(np.uint16), np.float16(x).view(np.uint16))


def test_ixsq_reader_rejects_other_quantizers_and_flat_files_still_load(tmp_path):
    p = str(tmp_path / "index")
    faiss_io.write_sq_fp16_index(p, np.ones((2, 4), np.float16), 0)
    raw = bytearray(open(p, "rb").read())
    raw[4 + 33:4 + 37] = struct.pack("<i", 0)  # qtype QT_8bit
    open(p, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match="qtype 0"):
        faiss_io.read_index(p)
    x = gauss(5, 8, 1)
    faiss_io.write_flat_index(p, x, faiss_io.METRIC_L2)
    y, m, kind = faiss_io.read_index(p)
    assert kind == faiss_io.FLAT and m == 1 and np.array_equal(y, x)
    d = str(tmp_path / "dir")
    faiss_io.write_index_dir(d, x, x, 0)
    assert faiss_io.read_index_dir(d, with_kind=True)[3] == faiss_io.FLAT
    assert len(faiss_io.read_index_dir(d)) == 3


def test_ixsq_against_real_faiss(tmp_path):
    """Pins the layout against a running faiss. Skips where the faiss wheel is not installed."""
    faiss = pytest.importorskip("faiss")
    x, q = gauss(40, 16, 3), gauss(5, 16, 4)
    idx = faiss.index_factory(16, "SQfp16", faiss.METRIC_INNER_PRODUCT)
    idx.add(x)
    p = str(tmp_path / "theirs")
    faiss.write_index(idx, p)
    y, m, kind = faiss_io.read_index(p)
    assert kind == faiss_io.SQFP16 and m == 0 and np.array_equal(y, np.float16(x))
    ours = str(tmp_path / "ours")
    faiss_io.write_sq_fp16_index(ours, np.float16(x), 0)
    back = faiss.read_index(ours)
    assert np.array_equal(back.search(q, 5)[1], idx.search(q, 5)[1])


# ---- B200VS host semantics -------------------------------------------------------------------------------------------------
def test_factory_and_dtype_validation():
    with pytest.raises(ValueError, match="flat"):
        B200VS(factory_string="SQ8")
    with pytest.raises(ValueError, match="flat"):
        B200VS(factory_string="SQbf16")
    with pytest.raises(ValueError, match="SQfp16"):
        B200VS(factory_string="SQfp16", dtype="bf16")
    assert B200VS(factory_string="SQfp16").dtype == "f16"
    assert B200VS(dtype="f16").dtype == "f16"


def test_f16_flat_store_rounds_once_and_ships_exact_queries_as_f16(fake_native, tmp_path):
    x = gauss(40, 16, 5)
    vs = B200VS(dtype="f16")
    d = str(tmp_path / "f")
    vs.index(None, x, d)
    assert vs.b2_index.dtype == nv.F16 and np.array_equal(vs.b2_index.vals, f16(x))
    assert np.array_equal(faiss_io.read_flat_index(f"{d}/index")[0], x)   # a Flat file keeps what faiss would: fp32
    got = vs.get_vectors_from_index(d, [2, 7, 11])
    assert got.dtype == np.float32 and np.array_equal(got, f16(x)[[2, 7, 11]])
    out = vs(got, 4)
    assert vs.b2_index.calls[-1][:2] == (np.dtype(np.uint16), nv.F16)
    D, I = oracle.knn(f16(x), got, 4, oracle.IP)
    assert np.array_equal(out.indices, I) and np.array_equal(out.distances, D)
    vs(got * np.float32(1.0 + 2.0 ** -13), 4)                            # no longer fp16-exact: fp32 queries
    assert vs.b2_index.calls[-1][:2] == (np.dtype(np.float32), nv.F32)


def test_sqfp16_store_semantics(fake_native, tmp_path):
    x, q = gauss(60, 16, 6), gauss(5, 16, 7)
    vs = B200VS(factory_string="SQfp16", metric=faiss_io.METRIC_L2)
    d = str(tmp_path / "sq")
    vs.index(None, x, d)
    y, m, kind = faiss_io.read_index(f"{d}/index")
    assert kind == faiss_io.SQFP16 and m == 1 and np.array_equal(y, np.float16(x))
    with open(f"{d}/vecs", "rb") as fp:
        assert np.array_equal(pickle.load(fp), x)
    # scores: the fp32 query, NOT rounded, against the fp16 rows
    out = vs(q, 6)
    assert vs.b2_index.calls[-1][:2] == (np.dtype(np.float32), nv.F32)
    D, I = oracle.knn(f16(x), q, 6, oracle.L2)
    assert np.array_equal(out.indices, I) and np.array_equal(out.distances, D)
    # get_vectors_from_index returns the ORIGINAL embeddings (faiss_vs.py:38-41), not the fp16 rows
    assert np.array_equal(vs.get_vectors_from_index(d, [3, 0, 59]), x[[3, 0, 59]])
    # ids= : FaissVS re-quantises originals[ids], i.e. the same fp16 rows: a subset search of the store
    sub = np.array([50, 3, 17, 4, 33])
    out = vs(q, 3, ids=sub.tolist())
    D, I = oracle.knn_subset(f16(x), q, 3, sub, oracle.L2)
    assert np.array_equal(out.indices, I) and np.array_equal(out.distances, D)
    # padding past the rows searched
    out = vs(q, 8, ids=sub.tolist())
    assert (out.indices[:, 5:] == -1).all() and (out.distances[:, 5:] == np.finfo(np.float32).max).all()


def test_sqfp16_kmeans_trains_on_the_originals(fake_native, tmp_path):
    rng = np.random.default_rng(8)
    x = (rng.standard_normal((80, 12)) * 3).astype(np.float32)
    vs = B200VS(factory_string="SQfp16")
    vs.index(None, x, str(tmp_path / "k"))
    ids = np.arange(0, 80, 2)
    a, c, _ = vs.kmeans(ids, 4, niter=5)
    wa, wc, _ = oracle.kmeans(np.ascontiguousarray(x[ids]), 4, niter=5)
    assert np.array_equal(a, wa) and np.array_equal(c, wc)
    assert FakeIndex.live == 1  # the temporary fp32 index was closed


def test_sqfp16_dedup_takes_the_asymmetric_reference_relation(fake_native, tmp_path, monkeypatch):
    import pandas as pd

    import lotus_b200 as lotus
    import lotus_b200.sem_ops.sem_dedup as sd

    rng = np.random.default_rng(9)
    base = gauss(6, 16, 10)
    emb = (base[rng.integers(0, 6, 30)] + rng.standard_normal((30, 16)).astype(np.float32) * 0.05).astype(np.float32)
    emb /= np.linalg.norm(emb, axis=1, keepdims=True)
    vals = [f"t{i}" for i in range(30)]
    vs = B200VS(factory_string="SQfp16")
    with pytest.raises(NotImplementedError):
        vs.threshold_pairs(0.5)
    monkeypatch.setattr(sd.nv, "connected_components", lambda n, pi, pj, device=0: oracle.connected_components(n, pi, pj))
    lotus.settings.configure(rm=lotus.TableRM({v: emb[i] for i, v in enumerate(vals)}), vs=vs, enable_cache=False)
    try:
        df = pd.DataFrame({"t": vals}).sem_index("t", str(tmp_path / "dd"))
        thr = 0.9
        kept = df.sem_dedup("t", thr)
    finally:
        lotus.settings.configure(rm=None, vs=None)
    # the relation the reference computes: x_i . fp16(x_j) > thr over the frame, then components over values
    D, I = oracle.knn_subset(f16(emb), emb, 30, np.arange(30), oracle.IP)
    qi, slot = np.nonzero(D > thr)
    pi, pj = qi, I[qi, slot]
    parent = list(range(30))

    def find(a):
        while parent[a] != a:
            a = parent[a]
        return a
    for a, b in zip(pi, pj):
        ra, rb = find(int(a)), find(int(b))
        if ra != rb:
            parent[max(ra, rb)] = min(ra, rb)
    survivors = [i for i in range(30) if find(i) == i]
    assert 0 < len(survivors) < 30
    assert kept["t"].tolist() == [vals[i] for i in survivors]


def test_out_of_range_corpus_and_directory_kind_mismatch(fake_native, tmp_path):
    x = gauss(10, 8, 11)
    bad = x.copy()
    bad[3, 2] = 7e4
    for vs in (B200VS(factory_string="SQfp16"), B200VS(dtype="f16")):
        with pytest.raises(ValueError, match="fp16"):
            vs.index(None, bad, str(tmp_path / "bad"))
    B200VS(factory_string="SQfp16").index(None, x, str(tmp_path / "sq"))
    B200VS().index(None, x, str(tmp_path / "flat"))
    with pytest.raises(ValueError, match="SQfp16"):
        B200VS().load_index(str(tmp_path / "sq"))
    with pytest.raises(ValueError, match="Flat"):
        B200VS(factory_string="SQfp16").load_index(str(tmp_path / "flat"))
    with pytest.raises(ValueError, match="metric"):
        B200VS(factory_string="SQfp16", metric=faiss_io.METRIC_L2).load_index(str(tmp_path / "sq"))
    vs = B200VS(factory_string="SQfp16")
    vs.load_index(str(tmp_path / "sq"))
    assert np.array_equal(vs.b2_index.vals, f16(x))
    assert np.array_equal(vs.get_vectors_from_index(str(tmp_path / "sq"), [1, 2]), x[[1, 2]])


def test_grid_values_are_exact_in_fp16():
    g = grid(50, 24, 12)
    assert np.array_equal(f16(g), g)


def test_reference_sq_replay_over_the_fake(fake_native, tmp_path):
    from sq_replay import replay_reference_sq_calls
    assert replay_reference_sq_calls(B200VS(factory_string="SQfp16"), str(tmp_path)) > 0
