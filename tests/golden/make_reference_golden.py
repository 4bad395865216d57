"""Generates tests/golden/reference_ops.json and tests/golden/reference_vs_calls.{json,npz} by running the REFERENCE's own
operator code.

    PYTHONHASHSEED=0 python tests/golden/make_reference_golden.py <checkout of lotus-data/lotus>

The reference (lotus-data/lotus @ 136ae4f4) is pure Python but cannot be imported as is: litellm, faiss,
sentence_transformers, backoff, ... are absent from this image. This script
  * satisfies every missing third-party import with an inert mock EXCEPT `faiss`, for which it installs a small stand-in
    module whose IndexFlat / Kmeans / read_index / write_index are backed by the oracle (oracle/faiss_flat.c) and by
    lotus_b200.faiss_io — i.e. the reference's control flow runs unmodified and only faiss's arithmetic is the restatement;
  * runs the reference's real `FaissVS` (lotus/vector_store/faiss_vs.py), `sem_index`, `sem_sim_join`, `sem_search`,
    `sem_dedup`, `sem_cluster_by` (lotus/sem_ops/*.py, lotus/utils.py) on small seeded inputs;
  * stores inputs and resulting DataFrames as JSON;
  * records every call those operators make on the vector store (index / load_index / get_vectors_from_index / search), with
    its arguments and FaissVS's answer (reference_vs_calls.*).
tests/test_reference_golden.py (CPU, oracle-backed test double) and tests/test_gpu_ops.py (B200VS) replay the scenarios
through lotus_b200's accessors and must reproduce the frames; tests/test_gpu_reference_dropin.py replays the recorded calls on
B200VS and must get FaissVS's answers. Nothing reads the reference at test time.
"""
import importlib.abc
import importlib.machinery
import json
import os
import sys
import tempfile
import types
import zlib
from unittest.mock import MagicMock

import numpy as np
import pandas as pd

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from lotus_b200 import faiss_io  # noqa: E402

MISSING = ("litellm", "sentence_transformers", "backoff", "qdrant_client", "weaviate", "tiktoken", "colbert", "gepa", "docker",
           "boto3", "sqlalchemy", "llama_index", "pymupdf", "fitz", "pptx", "bs4", "serpapi", "tavily", "arxiv")


class _MockFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, name, path, target=None):
        if name.split(".")[0] in MISSING:
            return importlib.machinery.ModuleSpec(name, self, is_package=True)
        return None

    def create_module(self, spec):
        m = MagicMock(name=spec.name)
        m.__path__, m.__spec__, m.__name__ = [], spec, spec.name
        return m

    def exec_module(self, module):
        pass


# ---- stand-in for the faiss wheel: control flow of the reference unchanged, arithmetic = the oracle --------------------
faiss = types.ModuleType("faiss")
faiss.METRIC_INNER_PRODUCT, faiss.METRIC_L2 = 0, 1


class _IndexFlat:
    def __init__(self, d, metric):
        self.d, self.metric_type = d, metric
        self.x = np.zeros((0, d), dtype=np.float32)

    @property
    def ntotal(self):
        return len(self.x)

    def add(self, x):
        self.x = np.concatenate([self.x, np.ascontiguousarray(x, dtype=np.float32)])

    def search(self, q, k):
        return oracle.knn(self.x, np.ascontiguousarray(q, dtype=np.float32), int(k), self.metric_type)


def _index_factory(d, factory_string, metric=0):
    assert factory_string == "Flat"
    return _IndexFlat(d, metric)


def _write_index(index, path):
    faiss_io.write_flat_index(path, index.x, index.metric_type)


def _read_index(path):
    x, metric = faiss_io.read_flat_index(path)
    idx = _IndexFlat(x.shape[1], metric)
    idx.add(x)
    return idx


class _Kmeans:
    def __init__(self, d, k, niter=25, verbose=False, **kw):
        self.d, self.k, self.niter = d, k, niter

    def train(self, x):
        x = np.ascontiguousarray(x, dtype=np.float32)
        _, cent, obj = oracle.kmeans(x, self.k, niter=self.niter)
        self.centroids = cent
        self.index = _IndexFlat(self.d, 1)
        self.index.add(cent)
        return float(obj[-1]) if len(obj) else 0.0


faiss.index_factory, faiss.write_index, faiss.read_index, faiss.Kmeans = _index_factory, _write_index, _read_index, _Kmeans
sys.modules["faiss"] = faiss
sys.meta_path.append(_MockFinder())
sys.path.insert(0, os.path.abspath(sys.argv[1]))
import lotus  # noqa: E402  (the REFERENCE package)
from lotus.models import RM  # noqa: E402
from lotus.vector_store import FaissVS  # noqa: E402


def hash_embed(docs, dim):
    out = np.empty((len(docs), dim), dtype=np.float32)
    for i, d in enumerate(docs):
        v = np.random.default_rng(zlib.crc32(str(d).encode("utf-8"))).standard_normal(dim).astype(np.float32)
        out[i] = v / np.linalg.norm(v)
    return out


class RefHashRM(RM):  # same embedding function as lotus_b200.HashRM
    def __init__(self, dim):
        super().__init__()
        self.dim = dim

    def _embed(self, docs):
        return hash_embed(docs, self.dim)


class RefTableRM(RM):
    def __init__(self, table):
        super().__init__()
        self.table = table

    def _embed(self, docs):
        return np.stack([np.asarray(self.table[d], dtype=np.float32) for d in docs]).astype(np.float32)


class RecordingFaissVS(FaissVS):
    """The reference's FaissVS, unchanged, with every call the operators make on it written down (arrays kept aside for the
    .npz; index directories relative to `root`)."""

    def __init__(self, root):
        super().__init__()
        self.root, self.calls, self.arrays = root, [], {}
        self.searching = False  # FaissVS.__call__ reads the subset through get_vectors_from_index: not an operator's call

    def _arr(self, a):
        name = f"a{len(self.arrays)}"
        self.arrays[name] = np.asarray(a)
        return name

    def _dir(self, d):
        return os.path.relpath(d, self.root)

    def index(self, docs, embeddings, index_dir, **kwargs):
        super().index(docs, embeddings, index_dir, **kwargs)
        self.calls.append({"op": "index", "dir": self._dir(index_dir), "docs": [str(v) for v in docs], "embeddings": self._arr(embeddings)})

    def load_index(self, index_dir):
        super().load_index(index_dir)
        self.calls.append({"op": "load_index", "dir": self._dir(index_dir)})

    def get_vectors_from_index(self, index_dir, ids):
        out = super().get_vectors_from_index(index_dir, ids)
        if self.searching:
            return out
        self.calls.append({"op": "get_vectors_from_index", "dir": self._dir(index_dir), "ids": [int(i) for i in ids],
                           "ids_type": "pandas.Index" if isinstance(ids, pd.Index) else "list", "out": self._arr(out)})
        return out

    def __call__(self, query_vectors, K, ids=None, **kwargs):
        self.searching = True
        try:
            out = super().__call__(query_vectors, K, ids=ids, **kwargs)
        finally:
            self.searching = False
        self.calls.append({"op": "search", "query": self._arr(query_vectors), "K": int(K), "ids": None if ids is None else [int(i) for i in ids],
                           "distances": self._arr(out.distances), "indices": self._arr(np.asarray(out.indices, dtype=np.int64))})
        return out


def frame_to_json(df):
    cols = [str(c) for c in df.columns]
    data = []
    for row in df.itertuples(index=False):
        data.append([float(np.float32(v)) if isinstance(v, (float, np.floating)) else (int(v) if isinstance(v, (int, np.integer)) else v)
                     for v in row])
    return {"index": [int(i) for i in df.index], "columns": cols, "data": data}


def main():
    out = {"_generated_by": "tests/golden/make_reference_golden.py against lotus-data/lotus @ 136ae4f4 (reference code) + oracle-backed faiss stand-in"}
    tmp = tempfile.mkdtemp()
    dim = 32
    vs = RecordingFaissVS(tmp)
    lotus.settings.configure(rm=RefHashRM(dim), vs=vs)

    left = pd.DataFrame({"a": [f"l{i}" for i in range(7)], "v": list(range(7))})
    right = pd.DataFrame({"b": [f"r{i}" for i in range(11)], "v": list(range(11))})
    right = right.sem_index("b", os.path.join(tmp, "r"))
    sc = {"dim": dim, "left": frame_to_json(left), "right": frame_to_json(right), "cases": []}
    for kw in ({"K": 3, "lsuffix": "_l", "rsuffix": "_r"}, {"K": 3, "lsuffix": "_l", "rsuffix": "_r", "keep_index": True},
               {"K": 1, "lsuffix": "x", "rsuffix": "y", "score_suffix": "_s"}):
        sc["cases"].append({"kwargs": kw, "right_rows": None, "out": frame_to_json(left.sem_sim_join(right, "a", "b", **kw))})
    sub = right[right["v"] % 2 == 0]
    for K in (4, 50):  # filtered right frame (ids=list(other.index)); K larger than the frame
        sc["cases"].append({"kwargs": {"K": K, "lsuffix": "_l", "rsuffix": "_r"}, "right_rows": [int(i) for i in sub.index],
                            "out": frame_to_json(left.sem_sim_join(sub, "a", "b", K=K, lsuffix="_l", rsuffix="_r"))})
    out["sim_join"] = sc

    docs = pd.DataFrame({"t": [f"doc{i}" for i in range(40)]}).sem_index("t", os.path.join(tmp, "s"))
    ss = {"dim": dim, "n": 40, "cases": []}
    for rows, K in ((None, 4), (None, 100), ([i for i in range(40) if i % 3 == 0], 5), ([5, 6, 7], 2)):
        frame = docs if rows is None else docs.loc[rows]
        res = frame.sem_search("t", "doc7", K=K, return_scores=True)
        ss["cases"].append({"rows": rows, "K": K, "query": "doc7", "out": frame_to_json(res)})
    out["search"] = ss

    vals = [f"v{i % 40}" for i in range(100)]
    dd = pd.DataFrame({"Text": vals}).sem_index("Text", os.path.join(tmp, "d"))
    kept = dd.sem_dedup("Text", threshold=0.5)
    out["dedup"] = {"dim": dim, "values": vals, "threshold": 0.5, "kept_values": kept["Text"].tolist(),
                    "note": "which value of a component survives depends on Python's set iteration order in the reference "
                            "(sem_dedup.py:58-84); only the partition / survivor count is comparable"}

    rng = np.random.default_rng(7)
    centers = rng.standard_normal((3, 16)).astype(np.float32) * 4
    names = [f"item{i}" for i in range(60)]
    table = {n: (centers[i % 3] + rng.standard_normal(16).astype(np.float32) * 0.3).astype(np.float32) for i, n in enumerate(names)}
    lotus.settings.configure(rm=RefTableRM(table))
    cf = pd.DataFrame({"name": names}).sem_index("name", os.path.join(tmp, "c"))
    cl = cf.sem_cluster_by("name", 3, niter=5)
    out["cluster"] = {"names": names, "table": {k: [float(x) for x in v] for k, v in table.items()}, "ncentroids": 3, "niter": 5,
                      "cluster_id": [int(c) for c in cl["cluster_id"]]}

    with open(os.path.join(HERE, "reference_ops.json"), "w") as f:
        json.dump(out, f)
    print("wrote tests/golden/reference_ops.json:", {k: (len(v["cases"]) if isinstance(v, dict) and "cases" in v else 1) for k, v in out.items() if not k.startswith("_")})
    with open(os.path.join(HERE, "reference_vs_calls.json"), "w") as f:
        json.dump({"_generated_by": out["_generated_by"], "calls": vs.calls}, f)
    np.savez_compressed(os.path.join(HERE, "reference_vs_calls.npz"), **vs.arrays)
    print(f"wrote tests/golden/reference_vs_calls.json + .npz: {len(vs.calls)} calls")


if __name__ == "__main__":
    main()
