"""df.sem_dedup(col, threshold) — lotus/sem_ops/sem_dedup.py:32-91.

Reference: self sim-join with K=len(df) (an N^2-row DataFrame), `_scores > threshold` (strict, :46), drop pairs whose
two TEXT VALUES are equal (:47), connected components over text values by DFS (:58-82), remove every value of a
component except one (:84-91, `isin` on values).
Here the all-pairs relation is produced by the streaming threshold kernel (never materialising N x N) and the
components by the device union-find; the value-based semantics are kept exactly. The reference's representative is
whichever node its DFS pops first from a Python set of string tuples (hash-seed dependent); ours is deterministic:
the value that appears first in the frame. Parity is therefore defined on the PARTITION and the survivor count."""
from __future__ import annotations

from typing import Any

import numpy as np
import pandas as pd

from .. import _native as nv
from ..cache import operator_cache
from ._common import register, resolve_rm_vs, validate_df


@register("sem_dedup")
class SemDedupByDataframe:
    def __init__(self, pandas_obj: Any):
        validate_df(pandas_obj)
        self._obj = pandas_obj

    @operator_cache
    def __call__(self, col_name: str, threshold: float) -> pd.DataFrame:
        rm, vs = resolve_rm_vs()
        try:
            col_index_dir = self._obj.attrs["index_dirs"][col_name]
        except KeyError:
            raise ValueError(f"Index directory for column {col_name} not found in DataFrame")
        if vs.index_dir != col_index_dir:
            vs.load_index(col_index_dir)
        assert vs.index_dir == col_index_dir

        n = len(self._obj)
        if n == 0:
            return self._obj
        rows = np.asarray(self._obj.index, dtype=np.int64)  # positions into the index (un-reset RangeIndex contract)
        pairs = None
        if hasattr(vs, "threshold_pairs"):
            try:
                pairs = vs.threshold_pairs(float(threshold))   # pairs over INDEX positions, i < j
            except NotImplementedError:
                pairs = None  # e.g. an SQfp16 store, whose relation is asymmetric: the reference relation below
            except nv.NativeError as e:
                if e.code in (nv.EINVAL, nv.ERANGE):  # e.g. an L2 index: the relation is defined on inner products
                    raise ValueError(e.msg) from e
                raise
        if pairs is not None:
            pi, pj = pairs
            # restrict to this frame's rows and translate to frame-local row numbers
            pos = np.full(int(max(rows.max(), pi.max() if len(pi) else 0, pj.max() if len(pj) else 0)) + 1, -1, dtype=np.int64)
            pos[rows] = np.arange(n)
            li, lj = pos[pi], pos[pj]
            ok = (li >= 0) & (lj >= 0)
            li, lj = li[ok], lj[ok]
        else:
            # any other VS (e.g. the reference's FaissVS), or a store without a symmetric all-pairs relation: the reference's own relation — every row against every row of the
            # frame through vs(..., K=n, ids=rows) (sem_dedup.py:45 via sem_sim_join.py:132-134), `_scores > threshold` (:46)
            qv = vs.get_vectors_from_index(col_index_dir, rows.tolist())
            out = vs(qv, n, ids=rows.tolist())
            sc = np.asarray(out.distances, dtype=np.float32).reshape(n, -1)
            ix = np.asarray([list(r) for r in out.indices], dtype=np.int64).reshape(n, -1)
            pos = np.full(int(rows.max()) + 1, -1, dtype=np.int64)
            pos[rows] = np.arange(n)
            qi, slot = np.nonzero((sc > threshold) & (ix >= 0))
            li, lj = qi.astype(np.int64), pos[ix[qi, slot]]
        # nodes are distinct text values, numbered in order of first appearance (sem_dedup.py:47,51-56); a missing value
        # (None / NaN, factorize code -1) never equals anything in the reference's `!=` / set logic either: it joins nothing
        codes, uniques = pd.factorize(self._obj[col_name], sort=False)
        ci, cj = codes[li], codes[lj]
        diff = (ci != cj) & (ci >= 0) & (cj >= 0)
        ci, cj = ci[diff], cj[diff]
        if len(uniques) == 0 or len(ci) == 0:
            return self._obj
        labels = nv.connected_components(len(uniques), ci, cj, getattr(vs, "device", 0))  # device union-find
        removed_codes = np.nonzero(labels != np.arange(len(uniques)))[0]
        removed_vals = uniques[removed_codes]
        return self._obj[~self._obj[col_name].isin(removed_vals)]
