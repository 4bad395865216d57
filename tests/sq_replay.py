"""Replay of tests/golden/reference_sq_vs_calls.* (make_reference_sq_golden.py): every vector-store call the reference's own
operators made on FaissVS(factory_string="SQfp16"), with FaissVS's answers. Same rules as helpers.replay_reference_vs_calls:
identical ids and score bits, and -1 padding past the rows searched where FaissVS wraps the pad to the last id."""
import json
import os

import numpy as np
import pandas as pd

from helpers import bits

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def replay_reference_sq_calls(vs, root):
    with open(os.path.join(GOLDEN, "reference_sq_vs_calls.json")) as f:
        calls = json.load(f)["calls"]
    arrays = np.load(os.path.join(GOLDEN, "reference_sq_vs_calls.npz"))
    rows = {}
    for n, c in enumerate(calls):
        where = (n, c["op"])
        if c["op"] == "index":
            emb = arrays[c["embeddings"]]
            vs.index(pd.Series(c["docs"]), emb, os.path.join(root, c["dir"]))
            rows[c["dir"]] = len(emb)
        elif c["op"] == "load_index":
            vs.load_index(os.path.join(root, c["dir"]))
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
