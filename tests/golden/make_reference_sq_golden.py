"""Generates tests/golden/reference_sq_vs_calls.{json,npz}: every call the REFERENCE's own operators (sem_index, sem_sim_join,
sem_search, sem_dedup, sem_cluster_by) make on the reference's unmodified FaissVS(factory_string="SQfp16"), with FaissVS's
answers.

    PYTHONHASHSEED=0 python tests/golden/make_reference_sq_golden.py <checkout of lotus-data/lotus>

It reuses make_reference_golden.py's import set-up (inert mocks for the missing third-party packages, an oracle-backed stand-in
for `faiss`) and adds "SQfp16" to the stand-in: IndexScalarQuantizer(d, QT_fp16) stores the rows rounded to fp16 (round to
nearest even, like faiss's F16C encoder) and scores fp32 queries exactly against them (the oracle over the fp16-widened rows);
write_index / read_index use the IxSQ layout of lotus_b200.faiss_io. tests/sq_replay.py replays the calls (CPU over the
oracle-backed fake in tests/test_f16_host.py, GPU through B200VS in tests/test_gpu_f16.py)."""
import json
import os
import sys
import tempfile

import numpy as np
import pandas as pd

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_reference_golden as base  # noqa: E402  (installs the faiss stand-in and imports the reference package)

faiss_io, lotus = base.faiss_io, base.lotus


class _IndexSQfp16(base._IndexFlat):
    def add(self, x):
        super().add(np.ascontiguousarray(x, dtype=np.float32).astype(np.float16).astype(np.float32))


_flat_factory = base.faiss.index_factory


def _index_factory(d, factory_string, metric=0):
    if factory_string == "SQfp16":
        return _IndexSQfp16(d, metric)
    return _flat_factory(d, factory_string, metric)


def _write_index(index, path):
    if isinstance(index, _IndexSQfp16):
        faiss_io.write_sq_fp16_index(path, index.x.astype(np.float16), index.metric_type)
    else:
        faiss_io.write_flat_index(path, index.x, index.metric_type)


def _read_index(path):
    x, metric, kind = faiss_io.read_index(path)
    idx = _IndexSQfp16(x.shape[1], metric) if kind == faiss_io.SQFP16 else base._IndexFlat(x.shape[1], metric)
    idx.add(x)
    return idx


base.faiss.index_factory, base.faiss.write_index, base.faiss.read_index = _index_factory, _write_index, _read_index


def main():
    tmp = tempfile.mkdtemp()
    dim = 32
    vs = base.RecordingFaissVS(tmp)
    vs.factory_string = "SQfp16"
    lotus.settings.configure(rm=base.RefHashRM(dim), vs=vs)

    left = pd.DataFrame({"a": [f"l{i}" for i in range(7)]})
    right = pd.DataFrame({"b": [f"r{i}" for i in range(11)]}).sem_index("b", os.path.join(tmp, "r"))
    left.sem_sim_join(right, "a", "b", K=3, lsuffix="_l", rsuffix="_r")
    sub = right[right.index % 2 == 0]
    left.sem_sim_join(sub, "a", "b", K=4, lsuffix="_l", rsuffix="_r")
    left = left.sem_index("a", os.path.join(tmp, "l"))             # the left column indexed too: its vectors come from an SQ store
    left.sem_sim_join(right, "a", "b", K=2, lsuffix="_l", rsuffix="_r")

    docs = pd.DataFrame({"t": [f"doc{i}" for i in range(40)]}).sem_index("t", os.path.join(tmp, "s"))
    docs.sem_search("t", "doc7", K=4)
    docs.loc[[i for i in range(40) if i % 3 == 0]].sem_search("t", "doc7", K=5)

    vals = [f"v{i % 40}" for i in range(100)]
    pd.DataFrame({"Text": vals}).sem_index("Text", os.path.join(tmp, "d")).sem_dedup("Text", threshold=0.5)

    rng = np.random.default_rng(7)
    centers = rng.standard_normal((3, 16)).astype(np.float32) * 4
    names = [f"item{i}" for i in range(60)]
    table = {n: (centers[i % 3] + rng.standard_normal(16).astype(np.float32) * 0.3).astype(np.float32) for i, n in enumerate(names)}
    lotus.settings.configure(rm=base.RefTableRM(table))
    pd.DataFrame({"name": names}).sem_index("name", os.path.join(tmp, "c")).sem_cluster_by("name", 3, niter=5)

    gen = ("tests/golden/make_reference_sq_golden.py against lotus-data/lotus @ 136ae4f4 (reference code, FaissVS('SQfp16')) "
           "+ oracle-backed faiss stand-in")
    with open(os.path.join(HERE, "reference_sq_vs_calls.json"), "w") as f:
        json.dump({"_generated_by": gen, "calls": vs.calls}, f)
    np.savez_compressed(os.path.join(HERE, "reference_sq_vs_calls.npz"), **vs.arrays)
    print(f"wrote tests/golden/reference_sq_vs_calls.json + .npz: {len(vs.calls)} calls")


if __name__ == "__main__":
    main()
