"""fp16 stores on the B200: one JSON line per case, with the card name and power limit read in the same call.

    python scripts/f16_timing.py [--reps 3]

C3 shape (100k queries x 1M rows x 768, K=32): fp16 store + fp16 queries against bf16 store + bf16 queries, alternating in one
process: filter ms (b2_last_filter_ms), queries/s, and a 256-query head+tail parity sample against the oracle.
C2 shape (10k fp32 queries x 1M x 768, K=10): B200VS-equivalent SQfp16 store (fp16 rows, fp32 queries) against an fp32 Flat
store: wall time, second-level (deferred) and fallback query counts, device bytes of the index."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from lotus_b200 import _native as nv  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # pragma: no cover
        return {"gpu": "unknown", "power_limit": "unknown", "error": str(e)}


def gauss(n, d, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, d), dtype=np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


def timed_search(idx, q, k, code):
    nv.stats_reset()
    t0 = time.perf_counter()
    D, I = idx.search(q, k, code)
    wall = time.perf_counter() - t0
    return D, I, wall, nv.stats(), idx.last_filter_ms()


def parity(xf, qf, D, I, k, metric, m=256):
    sel = np.r_[0:m // 2, len(qf) - m // 2:len(qf)]
    Do, Io = oracle.knn(xf, qf[sel], k, metric)
    return bool(np.array_equal(I[sel], Io) and np.array_equal(D[sel].view(np.uint32), Do.view(np.uint32)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    info = card()
    n, d, nq = 1_000_000, 768, 100_000
    x, q = gauss(n, d, 1), gauss(nq, d, 2)
    stores = {}
    for name, enc, dec, code in (("f16", nv.f32_to_f16_bits, nv.f16_bits_to_f32, nv.F16),
                                 ("bf16", nv.f32_to_bf16_bits, nv.bf16_bits_to_f32, nv.BF16)):
        xb, qb = enc(x), enc(q)
        stores[name] = (nv.Index(xb, code, 0), dec(xb), qb, dec(qb), code)
    for rep in range(a.reps):
        for name, (idx, xf, qb, qf, code) in stores.items():
            D, I, wall, st, fms = timed_search(idx, qb, 32, code)
            print(json.dumps({"case": "c3", "store": name, "queries": name, "rep": rep, "nq": nq, "n": n, "d": d, "k": 32,
                              "filter_ms": round(fms, 3), "wall_s": round(wall, 4), "qps": round(nq / wall),
                              "fallback_queries": st["fallback_queries"], "parity_head_tail_256": parity(xf, qf, D, I, 32, 0), **info}),
                  flush=True)
    for idx, *_ in stores.values():
        idx.close()
    q2 = gauss(10_000, d, 3)
    x16 = nv.f32_to_f16_bits(x)
    sq = nv.Index(x16, nv.F16, 0)
    flat = nv.Index(x, nv.F32, 0)
    for rep in range(a.reps):
        for name, idx, xf, nbytes in (("SQfp16", sq, nv.f16_bits_to_f32(x16) if rep == 0 else None, n * d * 2),
                                      ("Flat", flat, x if rep == 0 else None, n * d * 4)):
            D, I, wall, st, fms = timed_search(idx, q2, 10, nv.F32)
            row = {"case": "c2", "store": name, "queries": "f32", "rep": rep, "nq": len(q2), "n": n, "d": d, "k": 10,
                   "wall_s": round(wall, 4), "filter_ms": round(fms, 3), "deferred_queries": st["second_level_queries"],
                   "fallback_queries": st["fallback_queries"], "index_store_bytes": nbytes, **info}
            if xf is not None:
                row["parity_head_tail_256"] = parity(xf, q2, D, I, 10, 0)
            print(json.dumps(row), flush=True)
    sq.close()
    flat.close()


if __name__ == "__main__":
    main()
