#!/usr/bin/env python
"""bench.py — sem_sim_join queries/sec on the BASELINE.json headline configuration.

Workload (BASELINE.json configs[2], the one the metric is quoted on; it fits one GPU): 100k queries x 1M-row
index, 768-d bf16, K=32, synthetic L2-normalised Gaussian embeddings (corpus seed 0, queries seed 1). A "step" is
one pass of the hot path over the whole query batch: `VS.__call__` of the sim-join (fused tcgen05 filter + exact
finalize [+ all-gather + k-way merge when the index is row-sharded over N GPUs]).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...     # the CPU arm: faiss flat search on the host cores (real faiss when importable,
                                             # else the oracle port), plus the reference's own sem_sim_join operator around it
    python bench.py --config c2|c4|c5 ...    # the secondary BASELINE.json configurations, same contract (bench_secondary.py)
    python bench.py --dump-outputs DIR ...   # also write what the last timed step returned (scores.npy, ids.npy) under DIR

Prints ONE JSON line (rank 0). `value` = device-resident throughput; `e2e` = the plugin's own host-buffer call
(b2_index_search at N=1: pinned host queries in, host scores + ids out, H2D/D2H inside; at N>1 ShardedIndex.search_host: each
rank copies 1/N of the queries over PCIe, the ranks all-gather them over NVLink); `operator_e2e` = DataFrame in -> DataFrame
out through the pandas accessor (N=1); `roofline` is the tcgen05 filter kernel against the measured dense bf16 peak
(MEASURED_PEAKS.json); `cpu_baseline` is the CPU arm on a bounded sample of the same workload; `parity` compares the (merged)
GPU result with the canonical oracle on 256 queries at EVERY N and says which oracle ran ("faiss" when the wheel is importable).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the source tree may be read-only: leave no __pycache__ in it

BLOCK_ROWS = 1 << 16  # data is generated in fixed row blocks so every world size sees the same matrix
DUMP_BYTES = 64 << 20  # --dump-outputs budget


def env_int(name: str, default: int) -> int:
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def gen_rows_torch(torch, lo: int, hi: int, d: int, seed: int, device, dtype):
    """Rows [lo, hi) of the synthetic matrix: N(0,1) fp32, L2-normalised in fp32, cast to `dtype`."""
    out = torch.empty((hi - lo, d), dtype=dtype, device=device)
    b0, b1 = lo // BLOCK_ROWS, (hi - 1) // BLOCK_ROWS if hi > lo else -1
    for b in range(b0, b1 + 1):
        g = torch.Generator(device=device)
        g.manual_seed(seed * 1_000_003 + b)
        blk = torch.randn((BLOCK_ROWS, d), generator=g, device=device, dtype=torch.float32)
        blk = blk / blk.norm(dim=1, keepdim=True)
        s, e = max(lo, b * BLOCK_ROWS), min(hi, (b + 1) * BLOCK_ROWS)
        out[s - lo:e - lo] = blk[s - b * BLOCK_ROWS:e - b * BLOCK_ROWS].to(dtype)
    return out


def gen_rows_numpy(lo: int, hi: int, d: int, seed: int) -> np.ndarray:
    """CPU generator for the reference arm (different stream of random numbers, same distribution)."""
    out = np.empty((hi - lo, d), dtype=np.float32)
    b0, b1 = lo // BLOCK_ROWS, (hi - 1) // BLOCK_ROWS if hi > lo else -1
    for b in range(b0, b1 + 1):
        rng = np.random.default_rng(seed * 1_000_003 + b)
        blk = rng.standard_normal((BLOCK_ROWS, d), dtype=np.float32)
        blk /= np.linalg.norm(blk, axis=1, keepdims=True)
        s, e = max(lo, b * BLOCK_ROWS), min(hi, (b + 1) * BLOCK_ROWS)
        out[s - lo:e - lo] = blk[s - b * BLOCK_ROWS:e - b * BLOCK_ROWS]
    return out


def to_bf16_values(a: np.ndarray) -> np.ndarray:
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    r = (u + np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1))) & np.uint32(0xFFFF0000)  # RNE; inputs are finite
    return r.view(np.float32).reshape(a.shape)


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines: list[str] = []
        self.proc = None
        self.thread = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            assert self.proc is not None and self.proc.stdout is not None
            for line in self.proc.stdout:
                self.lines.append(line.strip())

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
                power.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(out_dir: str, scores, ids) -> None:
    """Writes what one search of the query batch hands its caller: scores[nq, k] as float32 (scores.npy) and ids[nq, k] as
    float64 (ids.npy; exact, the ids are below 2**53). Over DUMP_BYTES, a fixed seeded sample of query rows is written instead,
    in ascending order, with their positions in the batch (rows.npy, float64): the same rows for the same arguments, so two
    builds can be compared output for output."""
    import torch
    nq, k = scores.shape
    keep = DUMP_BYTES // (k * (4 + 8) + 8)
    os.makedirs(out_dir, exist_ok=True)
    if nq > keep:
        rows = np.sort(np.random.default_rng(0).choice(nq, size=keep, replace=False))
        sel = torch.from_numpy(rows).to(scores.device)
        scores, ids = scores[sel], ids[sel]
        np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "scores.npy"), scores.float().cpu().numpy())
    np.save(os.path.join(out_dir, "ids.npy"), ids.cpu().numpy().astype(np.float64))


def load_peaks() -> tuple[float, str]:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            pk = json.load(f)
        if "bf16_tflops_sustained" in pk:
            return float(pk["bf16_tflops_sustained"]), "measured bf16_tflops_sustained (MEASURED_PEAKS.json; kernel timed inside a long step)"
        return float(pk["bf16_tflops"]), "measured bf16_tflops (MEASURED_PEAKS.json)"
    except Exception:
        return 1590.0, "fallback 1.59 PFLOP/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


# ---- CPU arms ------------------------------------------------------------------------------------------------------------------
def faiss_probe() -> dict:
    """SURVEY §8c plan item 4 / BASELINE.md §3: if `import faiss` succeeds it becomes the primary oracle and the restatement is
    validated against it first. Returns {"oracle": "faiss"|"port", ...}."""
    try:
        import faiss  # type: ignore
    except Exception as exc:
        return {"oracle": "port", "faiss": f"not importable ({type(exc).__name__})",
                "note": "oracle/faiss_flat.c restates faiss 1.13; PARITY UNPINNED against a running faiss (DESIGN.md §7)"}
    import oracle
    out = {"oracle": "faiss", "faiss": getattr(faiss, "__version__", "?"), "omp_threads": faiss.omp_get_max_threads()}
    try:  # the restatement against the real thing on the committed golden inputs (tie-heavy grid set + Gaussian set)
        g = np.load(os.path.join(ROOT, "tests", "golden", "knn_golden.npz"))
        agree = {}
        for ds in ("grid", "gauss"):
            x, q = np.ascontiguousarray(g[f"{ds}_x"], dtype=np.float32), np.ascontiguousarray(g[f"{ds}_q"], dtype=np.float32)
            for name, metric, cls in (("ip", oracle.IP, faiss.IndexFlatIP), ("l2", oracle.L2, faiss.IndexFlatL2)):
                for kk in (1, 5, 32):
                    ix = cls(x.shape[1])
                    ix.add(x)
                    Df, If = ix.search(q, kk)
                    agree[f"{ds}_{name}_k{kk}"] = {"idx_equal": bool(np.array_equal(If, g[f"{ds}_{name}_k{kk}_I"])),
                                                   "max_abs_score_diff": float(np.abs(Df - g[f"{ds}_{name}_k{kk}_D"]).max())}
        out["golden_vs_faiss"] = agree
        out["golden_all_idx_equal"] = bool(all(v["idx_equal"] for v in agree.values()))
    except Exception as exc:  # pragma: no cover
        out["golden_vs_faiss"] = {"error": repr(exc)[:200]}
    return out


def cpu_arms(x: np.ndarray, q_pool: np.ndarray, k: int, requested: int, target_s: float) -> dict:
    """Times the CPU implementations of the flat search on a bounded sample (all host cores):
       - faiss.IndexFlatIP.search when the wheel is importable (kind "reference"),
       - the oracle port, cache-tiled and compiled for this host (orc_knn_tiled, -march=native),
       - numpy (OpenBLAS) sgemm + argpartition, what faiss's BLAS path does at the cache level.
    The first available of these, in that order, is the headline `value`; all are reported with their TFLOP/s."""
    import oracle
    oracle.build()
    cores = oracle.use_all_cores_native()
    n, d = x.shape
    fl_per_q = 2.0 * n * d
    arms = {}
    # calibrate the sample on the tiled port: one super-block per thread at least
    probe = min(max(256, 16 * cores), len(q_pool))
    oracle.knn_tiled(x[:50_000], q_pool[:probe], k, oracle.IP)
    t0 = time.perf_counter()
    oracle.knn_tiled(x, q_pool[:probe], k, oracle.IP)
    rate = probe / max(time.perf_counter() - t0, 1e-6)
    sample = requested if requested > 0 else int(min(max(int(rate * target_s) // 256 * 256, 256), len(q_pool)))
    sample = min(sample, len(q_pool))
    qs = np.ascontiguousarray(q_pool[:sample])
    t0 = time.perf_counter()
    Dt, It = oracle.knn_tiled(x, qs, k, oracle.IP)
    dt = time.perf_counter() - t0
    arms["port_tiled_native"] = {"queries_per_s": sample / dt, "tflops": fl_per_q * sample / dt / 1e12, "seconds": dt, "queries": sample,
                                 "what": f"oracle/faiss_flat.c orc_knn_tiled (fp32 FMA micro-kernel, 256-row corpus tiles, OpenMP x{cores}, {oracle.native_flags()})"}
    s2 = min(sample, max(256, int(sample // 4)))
    try:
        t0 = time.perf_counter()
        Ds, Is = oracle.knn_sgemm(x, qs[:s2], k, oracle.IP)
        dt2 = time.perf_counter() - t0
        arms["numpy_sgemm_argpartition"] = {"queries_per_s": s2 / dt2, "tflops": fl_per_q * s2 / dt2 / 1e12, "seconds": dt2, "queries": s2,
                                            "what": "numpy (OpenBLAS) sgemm 2048 x 65536 blocks + argpartition + merge",
                                            "same_topk_sets_as_port": float(np.mean([len(set(a) & set(b)) / k for a, b in zip(Is, It[:s2])]))}
    except Exception as exc:  # pragma: no cover
        arms["numpy_sgemm_argpartition"] = {"error": repr(exc)[:200]}
    kind, head = "port", "port_tiled_native"
    try:
        import faiss  # type: ignore
        faiss.omp_set_num_threads(cores)
        ix = faiss.IndexFlatIP(d)
        ix.add(x)
        ix.search(qs[:64], k)
        t0 = time.perf_counter()
        Df, If = ix.search(qs, k)
        dtf = time.perf_counter() - t0
        arms["faiss_IndexFlatIP"] = {"queries_per_s": sample / dtf, "tflops": fl_per_q * sample / dtf / 1e12, "seconds": dtf, "queries": sample,
                                     "what": f"faiss {getattr(faiss, '__version__', '?')} IndexFlatIP.search, omp x{faiss.omp_get_max_threads()}",
                                     "idx_equal_to_port": bool(np.array_equal(If, It))}
        kind, head = "reference", "faiss_IndexFlatIP"
    except Exception:
        pass
    return {"value": arms[head]["queries_per_s"], "unit": "queries/s", "cores": cores, "kind": kind, "arm": head, "host": oracle.cpu_budget(),
            "sample": f"{arms[head]['queries']} of the queries x full {n}-row index, once ({arms[head]['seconds']:.1f} s): {arms[head]['what']}",
            "arms": arms, "_sample": sample, "_I": It, "_D": Dt}


def reference_operator_leg(args, x: np.ndarray, q: np.ndarray, k: int) -> dict:
    """Operator scope of the reference arm (SURVEY §8d-ii): the reference's UNMODIFIED sem_index + sem_sim_join
    (lotus/sem_ops/sem_sim_join.py:96-166 incl. its pickle re-reads, Python remap loop and two pandas joins) over its own FaissVS,
    with faiss = the real wheel when importable, else a stand-in whose IndexFlat.search is the timed CPU port. Left frame = a
    bounded sample of the queries, right frame = the full index."""
    import tempfile
    import types

    import pandas as pd
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle
    import refpkg
    from lotus_b200 import faiss_io
    stand_in = None
    try:
        import faiss  # type: ignore  # noqa: F401
    except Exception:
        stand_in = types.ModuleType("faiss")
        stand_in.METRIC_INNER_PRODUCT, stand_in.METRIC_L2 = 0, 1

        class _IndexFlat:
            def __init__(self, dd, metric):
                self.d, self.metric_type, self.x = dd, metric, np.zeros((0, dd), dtype=np.float32)

            @property
            def ntotal(self):
                return len(self.x)

            def add(self, v):
                v = np.ascontiguousarray(v, dtype=np.float32)
                self.x = v if len(self.x) == 0 else np.concatenate([self.x, v])

            def search(self, qq, kk):
                return oracle.knn_tiled(self.x, np.ascontiguousarray(qq, dtype=np.float32), int(kk), self.metric_type)

        def _factory(dd, fs, metric=0):
            return _IndexFlat(dd, metric)

        def _write(index, path):
            faiss_io.write_flat_index(path, index.x, index.metric_type)

        def _read(path):
            xx, metric = faiss_io.read_flat_index(path)
            ix = _IndexFlat(xx.shape[1], metric)
            ix.add(xx)
            return ix

        stand_in.index_factory, stand_in.write_index, stand_in.read_index = _factory, _write, _read
    lotus, faiss_kind = refpkg.import_reference(stand_in)
    if lotus is None:
        return {"unavailable": faiss_kind}
    from lotus.models import RM
    from lotus.vector_store import FaissVS

    class Precomputed(RM):
        def __init__(self):
            super().__init__()
            self.next = None

        def _embed(self, docs):
            return self.next

    rm = Precomputed()
    lotus.settings.configure(rm=rm, vs=FaissVS())
    left = pd.DataFrame({"article": [f"a{i}" for i in range(len(q))]})
    right = pd.DataFrame({"category": [f"c{i}" for i in range(len(x))]})
    with tempfile.TemporaryDirectory() as tmp:
        t0 = time.perf_counter()
        rm.next = q
        left = left.sem_index("article", os.path.join(tmp, "l"))
        rm.next = x
        right = right.sem_index("category", os.path.join(tmp, "r"))
        t_index = time.perf_counter() - t0
        t0 = time.perf_counter()
        out = left.sem_sim_join(right, "article", "category", K=k)
        t_join = time.perf_counter() - t0
    return {"value": len(q) / t_join, "unit": "queries/s", "seconds": t_join, "rows_out": int(len(out)), "left_rows": len(q), "right_rows": len(x),
            "sem_index_seconds_both_frames": t_index, "faiss": faiss_kind,
            "what": "reference lotus/sem_ops/sem_sim_join.py + lotus/vector_store/faiss_vs.py, unmodified (baseline/_ref)"}


def run_reference(args) -> None:
    """CPU arm of the headline config: faiss flat search on the host cores (real faiss when importable, else the oracle port,
    cache-tiled, -march=native), K timed steps each over a bounded sample of the workload; plus the reference's own operator
    (DataFrame -> DataFrame) once. Rank 0 only."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    import oracle
    oracle.build()
    n, d, k = args.n, args.d, args.k
    t0 = time.time()
    x = to_bf16_values(gen_rows_numpy(0, n, d, 0))
    q_pool = to_bf16_values(gen_rows_numpy(0, min(16384, args.nq), d, 1))
    gen_s = time.time() - t0
    probe = faiss_probe()
    arms = cpu_arms(x, q_pool, k, args.cpu_sample, 8.0)  # every step ~8 s of all host cores: W + K steps end within minutes
    sample = arms["_sample"]
    q = np.ascontiguousarray(q_pool[:sample])
    use_faiss = arms["kind"] == "reference"
    if use_faiss:
        import faiss  # type: ignore
        ix = faiss.IndexFlatIP(d)
        ix.add(x)
        step = lambda: ix.search(q, k)  # noqa: E731
    else:
        step = lambda: oracle.knn_tiled(x, q, k, oracle.IP)  # noqa: E731
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    val = sample / dt
    op = None
    if not args.no_operator:
        try:
            op = reference_operator_leg(args, x, np.ascontiguousarray(q_pool[:min(sample, 4096)]), k)
        except Exception as exc:  # never lose the line over the secondary leg
            op = {"error": repr(exc)[:300]}
    for key in ("_sample", "_I", "_D"):
        arms.pop(key, None)
    arms.update({"value": val, "sample": f"{sample} queries x full {n}-row index per step: {arms['arms'][arms['arm']]['what']}"})
    line = {
        "impl": "reference", "metric": "sem_sim_join queries/sec (1M x 768, K=32)", "value": val, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (bf16 values)", "data": "synthetic",
        # same keys and workload string as the B200 arm's `config`; what is specific to this run sits in `reference_run`
        "config": {"workload": f"sem_sim_join {args.nq} queries x {n} index, {d}-d bf16, K={k} (BASELINE.json configs[2])", "nq": args.nq,
                   "n": n, "d": d, "k": k, "parallelism": f"{arms['cores']} host threads (no GPU)", "l2_policy": "n/a (CPU arm)"},
        "reference_run": {"sample_queries_per_step": sample, "datagen_s": round(gen_s, 1), "tflops": 2.0 * n * d * val / 1e12,
                          "data": "same generator, distribution and seeds as the B200 arm (numpy stream instead of the CUDA one)"},
        "cpu_baseline": arms, "oracle": probe,
        "e2e": {"value": val, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "operator_e2e": op,
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def operator_leg(torch, nv, corpus, queries, k: int, reps: int = 2) -> dict:
    """Operator scope on the B200 (SURVEY §8d-ii): DataFrame in -> DataFrame out through the pandas accessor
    (lotus_b200/sem_ops/sem_sim_join.py: same control flow as the reference's, B200VS underneath), next to the VS boundary."""
    import tempfile

    import pandas as pd

    import lotus_b200 as lotus

    class Precomputed(lotus.RM):
        def __init__(self):
            super().__init__()
            self.next = None

        def _embed(self, docs):
            return self.next

        def __call__(self, docs):
            return self.next

    rm = Precomputed()
    vs = lotus.B200VS(dtype="bf16", device=corpus.device.index or 0)
    lotus.settings.configure(rm=rm, vs=vs, enable_cache=False)
    nq, n = queries.shape[0], corpus.shape[0]
    left = pd.DataFrame({"article": [f"a{i}" for i in range(nq)]})
    right = pd.DataFrame({"category": [f"c{i}" for i in range(n)]})
    try:
        with tempfile.TemporaryDirectory() as tmp:
            t0 = time.perf_counter()
            rm.next = queries
            left = left.sem_index("article", os.path.join(tmp, "l"))
            rm.next = corpus
            right = right.sem_index("category", os.path.join(tmp, "r"))
            t_index = time.perf_counter() - t0
            times = []
            nv.stats_reset()
            for _ in range(reps + 1):
                t0 = time.perf_counter()
                out = left.sem_sim_join(right, "article", "category", K=k)
                times.append(time.perf_counter() - t0)
            st = nv.stats()
            best = min(times[1:])
            return {"value": nq / best, "unit": "queries/s", "seconds": best, "all_reps_s": [round(t, 4) for t in times], "rows_out": int(len(out)),
                    "sem_index_seconds_both_frames": t_index, "fallback_queries": int(st["fallback_queries"]),
                    "what": "df.sem_sim_join(other, ...) over B200VS: get_vectors_from_index (device gather) -> b2_index_search(ids=) -> frame assembly"}
    finally:
        vs.close()
        lotus.settings.configure(rm=None, vs=None)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=str, default="c3", choices=["c3", "c2", "c4", "c5"],
                    help="c3 = the headline (BASELINE.json configs[2]); c2 / c4 / c5 = the secondary configurations")
    ap.add_argument("--nq", "--queries", dest="nq", type=int, default=100_000)
    ap.add_argument("--n", "--corpus-rows", dest="n", type=int, default=1_000_000)
    ap.add_argument("--d", type=int, default=768)
    ap.add_argument("--k", type=int, default=32)
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries per CPU-baseline step (0 = about 8-15 s of the host cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-operator", action="store_true", help="skip the DataFrame -> DataFrame leg")
    ap.add_argument("--parity-queries", type=int, default=256)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the scores and ids the last timed step computed as DIR/<name>.npy (headline B200 run only)")
    args, extra = ap.parse_known_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != "c3" or args.impl != "b200"):
        ap.error("--dump-outputs is supported by the headline B200 run (--config c3 --impl b200)")
    if args.warmup < 3:
        args.warmup = 3
    if args.config != "c3":
        import bench_secondary
        bench_secondary.main(args, extra)
        return
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    from lotus_b200 import _native as nv
    from lotus_b200.distributed import ShardedIndex, shard_bounds

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=device)
    nv.require_device()

    nq, n, d, k = args.nq, args.n, args.d, args.k
    lo, hi = shard_bounds(n, world, rank)
    corpus = gen_rows_torch(torch, lo, hi, d, 0, device, torch.bfloat16)
    queries = gen_rows_torch(torch, 0, nq, d, 1, device, torch.bfloat16)
    index = ShardedIndex(corpus, lo, nv.METRIC_IP)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item()) / steps

    filt_ms: list[float] = []
    last_out: list = []  # (scores, ids) of the latest step, for --dump-outputs

    def step_dev():
        last_out[:] = index.search(queries, k)
        filt_ms.append(index.last_filter_ms())

    # ---- device-resident throughput --------------------------------------------------------------------------------
    for _ in range(args.warmup):
        step_dev()
    filt_ms.clear()
    nv.stats_reset()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_step = timed(step_dev, args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last_out)
    last_out.clear()
    st = nv.stats()
    launches_per_step = st["launches"] / max(args.steps, 1) + (1 if world > 1 else 0)  # + the all-gather kernel is NCCL's
    fallback_q = st["fallback_queries"]
    kernel_ms = float(np.mean(filt_ms)) if filt_ms else float("nan")
    kernel_ms_ranks = [kernel_ms]
    if world > 1:  # the all-gather makes every step wait for the slowest rank: report the spread
        t = torch.tensor([kernel_ms], device=device, dtype=torch.float64)
        allk = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allk, t)
        kernel_ms_ranks = [float(a.item()) for a in allk]
    phases = None
    if world > 1:  # one extra, untimed step with per-phase CUDA events (B2_SHARD_TIMING): what the non-filter time is made of
        os.environ["B2_SHARD_TIMING"] = "1"
        index.search(queries, k)
        os.environ.pop("B2_SHARD_TIMING", None)
        phases = {kk: round(v, 3) for kk, v in getattr(index, "last_phase_ms", {}).items()}

    # ---- end to end through the plugin's own call: host (pinned) queries in, host results out, every step -----------------
    q_host = queries.cpu().pin_memory()
    out_s_host = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    out_i_host = torch.empty((nq, k), dtype=torch.int64).pin_memory()
    h2d = q_host.numel() * q_host.element_size()
    d2h = out_s_host.numel() * 4 + out_i_host.numel() * 8
    if world == 1:
        # b2_index_search, the C-ABI call B200VS.__call__ makes: it copies q H2D, searches, copies scores + ids D2H and returns
        # when they are in host memory (its own stream: timed by the host clock around the synchronous call)
        import ctypes
        L = nv.lib()
        qb = q_host.view(torch.int16).numpy().view(np.uint16)
        Dh, Ih = out_s_host.numpy(), out_i_host.numpy()

        def step_e2e():
            nv.check(L.b2_index_search(index.index.handle, qb.ctypes.data_as(ctypes.c_void_p), nq, nv.BF16, k, None, 0,
                                       Dh.ctypes.data_as(ctypes.c_void_p), Ih.ctypes.data_as(ctypes.c_void_p)))

        for _ in range(2):
            step_e2e()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        ms_e2e = (time.perf_counter() - t0) / args.steps * 1e3
        e2e_api = "b2_index_search (C-ABI, host buffers in and out: the call B200VS.__call__ makes); host wall clock around the synchronous call"
        h2d_rank = h2d
    else:
        def step_e2e():
            index.search_host(q_host, k, out_s_host if rank == 0 else None, out_i_host if rank == 0 else None)

        for _ in range(2):
            step_e2e()
        ms_e2e = timed(step_e2e, args.steps)
        e2e_api = ("ShardedIndex.search_host: every rank copies 1/N of the pinned host queries H2D, NCCL all-gather of the query slices, "
                   "sharded search, rank 0 copies the merged result D2H; CUDA events, max over ranks")
        h2d_rank = h2d // world

    # ---- roofline of the dominant kernel (the tcgen05 filter), per rank-0 launch --------------------------------------
    peak_tf, peak_src = load_peaks()
    flops_launch = 2.0 * nq * (hi - lo) * d  # algorithmic: 2*N_local*d per query (SURVEY §8d)
    achieved_tf = flops_launch / (kernel_ms * 1e-3) / 1e12 if kernel_ms == kernel_ms and kernel_ms > 0 else None
    traffic = None
    try:  # DRAM bytes of one launch of this kernel on this shape, from the committed `ncu --set full` capture
        with open(os.path.join(ROOT, "profiles", "filter_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("nq") == nq and tj.get("n_local") == hi - lo and tj.get("d") == d:
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
    except Exception:
        traffic = None
    roofline = {"bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": (achieved_tf / peak_tf) if achieved_tf else None, "traffic": traffic,
                "kernel": "knn_filter_kernel<KP=64,IP,bf16,cta_group::2>", "kernel_ms": kernel_ms, "peak_source": peak_src,
                "kernel_ms_per_rank": [round(v, 3) for v in kernel_ms_ranks],
                "algorithmic_flops_per_launch": flops_launch,
                "hbm_floor_ms": ((hi - lo) * d * 2 + nq * d * 2 + nq * k * 12) / 6.4843e12 * 1e3}

    # ---- parity at every N: the (merged) result of 256 queries against the canonical oracle, indices and score bits ----------
    parity = None
    npar = max(0, min(args.parity_queries, nq))
    # half of the sample from the head of the batch, half from its tail: the filter schedules the leading query units (whole
    # waves) and the trailing ones (split remainder) differently, and the sample is searched as part of the FULL batch
    par_rows = None
    if npar:
        head = npar - npar // 2
        par_rows = torch.cat([torch.arange(0, head, device=device), torch.arange(nq - npar // 2, nq, device=device)])
        s_all, i_all = index.search(queries, k)
        s_par, i_par = s_all[par_rows].contiguous(), i_all[par_rows].contiguous()
        del s_all, i_all
    else:
        s_par, i_par = None, None
    cpu_baseline = None
    operator_e2e = None
    if rank == 0:
        import oracle
        oracle.build()
        oracle.use_all_cores()
        xs_dev = corpus if world == 1 else gen_rows_torch(torch, 0, n, d, 0, device, torch.bfloat16)
        xs = xs_dev.float().cpu().numpy()
        del xs_dev
        probe = faiss_probe()
        if npar:
            qs = queries[par_rows].float().cpu().numpy()
            t0 = time.perf_counter()
            Do, Io = oracle.knn(xs, qs, k, oracle.IP)
            Ig, Dg = i_par.cpu().numpy(), s_par.cpu().numpy()
            parity = {"queries": npar, "sample": "first %d and last %d queries of the batch, taken from a search of the WHOLE batch" % (npar - npar // 2, npar // 2),
                      "oracle": probe["oracle"], "oracle_detail": probe,
                      "against": "oracle.knn (canonical fp64-accumulated score, faiss heap tie rule) on the full index",
                      "idx_bit_exact_vs_oracle": bool(np.array_equal(Ig, Io)),
                      "score_bit_exact_vs_oracle": bool(np.array_equal(Dg.view(np.uint32), Do.view(np.uint32))),
                      "recall_at_k": float(np.mean([len(set(a) & set(b)) / k for a, b in zip(Ig, Io)])),
                      "rows_differing": int((Ig != Io).any(axis=1).sum()), "oracle_seconds": round(time.perf_counter() - t0, 1)}
            if probe["oracle"] == "faiss":
                import faiss  # type: ignore
                ix = faiss.IndexFlatIP(d)
                ix.add(xs)
                Df, If = ix.search(qs, k)
                parity.update({"idx_equal_to_faiss": bool(np.array_equal(Ig, If)), "max_abs_score_diff_vs_faiss": float(np.abs(Dg - Df).max()),
                               "recall_at_k_vs_faiss": float(np.mean([len(set(a) & set(b)) / k for a, b in zip(Ig, If)]))})
        if world == 1 and not args.no_cpu_baseline:
            q_pool = queries[:min(16384, nq)].float().cpu().numpy()
            cpu_baseline = cpu_arms(xs, q_pool, k, args.cpu_sample, 12.0)
            sample, Ic = cpu_baseline.pop("_sample"), cpu_baseline.pop("_I")
            cpu_baseline.pop("_D")
            s_dev, i_dev = index.search(queries[:sample].contiguous(), k)
            if parity is not None:  # recall@K of the GPU result against the fp32 CPU flat search on the whole CPU sample
                parity["recall_at_k_vs_cpu_flat"] = float(np.mean([len(set(a) & set(b)) / k for a, b in zip(i_dev.cpu().numpy(), Ic)]))
                parity["cpu_flat_sample_queries"] = sample
        del xs
    if world == 1 and rank == 0 and not args.no_operator:
        try:
            operator_e2e = operator_leg(torch, nv, corpus, queries, k)
        except Exception as exc:  # never lose the bench line over the secondary leg
            operator_e2e = {"error": repr(exc)[:300]}

    if rank == 0:
        line = {
            "metric": "sem_sim_join queries/sec (1M x 768, K=32)", "value": nq / (ms_step * 1e-3), "unit": "queries/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"sem_sim_join {nq} queries x {n} index, {d}-d bf16, K={k} (BASELINE.json configs[2])",
                       "nq": nq, "n": n, "d": d, "k": k, "parallelism": f"index row-sharded x{world}",
                       "l2_policy": "inputs exceed L2 (corpus shard %.0f MB + queries %.0f MB vs 126 MB L2)" %
                                    ((hi - lo) * d * 2 / 1e6, nq * d * 2 / 1e6)},
            "e2e": {"value": nq / (ms_e2e * 1e-3), "unit": "queries/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": h2d_rank, "d2h_bytes_per_step": d2h, "api": e2e_api},
            "operator_e2e": operator_e2e,
            "gpu_launches": int(round(launches_per_step * args.steps)),
            "gpu_launches_per_step": launches_per_step,
            "fallback_queries": int(fallback_q),
            "roofline": roofline,
            "shard_phases_ms": phases,
            "cpu_baseline": cpu_baseline,
            "parity": parity,
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    index.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
