"""oracle — TEST INFRASTRUCTURE ONLY (see oracle/faiss_flat.c header).

CPU restatement of the faiss-cpu 1.13 algorithms behind the reference's hot path
(lotus/vector_store/faiss_vs.py:22-77, lotus/utils.py:61-65). PARITY UNPINNED: faiss itself is
not available in this image (nor on the GPU box) and the reference holds no golden vectors for this
path, so the restatement is pinned only against hand-derived known answers (tests/golden/) and
independent numpy cross-checks. bench.py `faiss_probe()` / `cpu_arms()` switch to the real wheel the
day `import faiss` succeeds and print the comparison with this restatement.

Besides the canonical oracle (`knn`, `kmeans`, ...: portable build, -ffp-contract=off) this package holds
the TIMED CPU arms of bench.py: `knn_tiled` (cache-tiled fp32 FMA search, compiled on the host with
-march=native), `knn_sgemm` (numpy/OpenBLAS sgemm + argpartition) and `cpu_budget()` (affinity capped by
the cgroup CPU quota).

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this package.
Nothing under lotus_b200/ imports it.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "faiss_flat.c")
_LIB = os.path.join(_HERE, "liborc.so")

IP, L2 = 0, 1
CANONICAL, F32_SEQ, F32_FAST = 0, 1, 2


def build(force: bool = False) -> str:
    """gcc-compile oracle/faiss_flat.c into oracle/liborc.so (git-ignored, travels with gpurun)."""
    if not force and os.path.exists(_LIB) and os.path.getmtime(_LIB) >= os.path.getmtime(_SRC):
        return _LIB
    cmd = ["gcc", "-O3", "-march=x86-64-v3", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared",
           "-o", _LIB, _SRC, "-lm"]
    try:
        subprocess.run(cmd, check=True, capture_output=True, text=True)
    except subprocess.CalledProcessError as e:  # pragma: no cover
        sys.stderr.write(e.stderr)
        raise
    return _LIB


_NATIVE = os.path.join(_HERE, "liborc_native.so")
_native_lib = None
_native_flags = None


def native_lib():
    """The same source compiled ON THIS HOST with -march=native (AVX-512 where the host has it) and fp contraction, for the TIMED
    CPU arm only (bench.py): the portable liborc.so is built in the build container for x86-64-v3 so that it runs anywhere and
    keeps -ffp-contract=off for the canonical scorer. Falls back to the portable library when gcc is not available here.
    Compiled (about 2 s) into a private temporary directory that is removed once the library is loaded: the source tree may be
    read-only, and nothing is left behind."""
    global _native_lib, _native_flags
    if _native_lib is not None:
        return _native_lib
    flags = ["-O3", "-march=native", "-mtune=native", "-ffp-contract=fast", "-funroll-loops"]
    try:
        import shutil
        import tempfile
        tmp = tempfile.mkdtemp(prefix="liborc_native_")
        try:
            path = os.path.join(tmp, "liborc_native.so")
            subprocess.run(["gcc", *flags, "-fopenmp", "-fPIC", "-shared", "-o", path, _SRC, "-lm"], check=True, capture_output=True, text=True)
            L = ctypes.CDLL(path)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        _native_flags = " ".join(flags)
    except Exception:
        L = lib()
        _native_flags = "-O3 -march=x86-64-v3 (portable build; native build unavailable)"
    f32p = ctypes.POINTER(ctypes.c_float)
    i64p = ctypes.POINTER(ctypes.c_int64)
    L.orc_knn_tiled.restype = ctypes.c_int
    L.orc_knn_tiled.argtypes = [f32p, ctypes.c_int64, ctypes.c_int, f32p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, f32p, i64p]
    L.orc_num_threads.restype = ctypes.c_int
    L.orc_set_num_threads.argtypes = [ctypes.c_int]
    L.orc_set_num_threads.restype = None
    _native_lib = L
    return L


def native_flags() -> str:
    native_lib()
    return _native_flags


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB) or (os.path.exists(_SRC) and os.path.getmtime(_LIB) < os.path.getmtime(_SRC)):
            build()
        L = ctypes.CDLL(_LIB)
        f32p = ctypes.POINTER(ctypes.c_float)
        i64p = ctypes.POINTER(ctypes.c_int64)
        i32p = ctypes.POINTER(ctypes.c_int32)
        u32p = ctypes.POINTER(ctypes.c_uint32)
        L.orc_num_threads.restype = ctypes.c_int
        L.orc_set_num_threads.argtypes = [ctypes.c_int]
        L.orc_set_num_threads.restype = None
        L.orc_dot_canonical.restype = ctypes.c_float
        L.orc_dot_canonical.argtypes = [f32p, f32p, ctypes.c_int]
        L.orc_l2_canonical.restype = ctypes.c_float
        L.orc_l2_canonical.argtypes = [f32p, f32p, ctypes.c_int]
        L.orc_norm2_canonical_f64.restype = ctypes.c_double
        L.orc_norm2_canonical_f64.argtypes = [f32p, ctypes.c_int]
        L.orc_scores.restype = None
        L.orc_scores.argtypes = [f32p, ctypes.c_int64, ctypes.c_int, f32p, ctypes.c_int64, ctypes.c_int,
                                 ctypes.c_int, f32p]
        L.orc_knn.restype = ctypes.c_int
        L.orc_knn.argtypes = [f32p, ctypes.c_int64, ctypes.c_int, f32p, ctypes.c_int64, ctypes.c_int,
                              ctypes.c_int, ctypes.c_int, f32p, i64p]
        L.orc_knn_blocked.restype = ctypes.c_int
        L.orc_knn_blocked.argtypes = [f32p, ctypes.c_int64, ctypes.c_int, f32p, ctypes.c_int64, ctypes.c_int,
                                      ctypes.c_int, f32p, i64p]
        L.orc_knn_tiled.restype = ctypes.c_int
        L.orc_knn_tiled.argtypes = [f32p, ctypes.c_int64, ctypes.c_int, f32p, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                    ctypes.c_int, f32p, i64p]
        L.orc_threshold_pairs.restype = ctypes.c_int64
        L.orc_threshold_pairs.argtypes = [f32p, ctypes.c_int64, ctypes.c_int, ctypes.c_float, i64p, i64p,
                                          ctypes.c_int64]
        L.orc_mt_fill.restype = None
        L.orc_mt_fill.argtypes = [ctypes.c_uint32, u32p, ctypes.c_int]
        L.orc_rand_perm.restype = None
        L.orc_rand_perm.argtypes = [i32p, ctypes.c_int64, ctypes.c_int64]
        L.orc_compute_centroids.restype = None
        L.orc_compute_centroids.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int64, f32p, i64p, f32p, f32p]
        L.orc_split_clusters.restype = ctypes.c_int
        L.orc_split_clusters.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int64, f32p, f32p]
        L.orc_kmeans.restype = ctypes.c_int
        L.orc_kmeans.argtypes = [f32p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64,
                                 ctypes.c_int, ctypes.c_int, i64p, f32p, f32p]
        _lib = L
    return _lib


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a: np.ndarray, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


def num_threads() -> int:
    return int(lib().orc_num_threads())


def use_all_cores() -> int:
    """Give OpenMP every core this process may run on, whatever OMP_NUM_THREADS said (torchrun sets it to 1)."""
    lib().orc_set_num_threads(cpu_budget()["threads"])
    return num_threads()


def to_bf16_f32(a) -> np.ndarray:
    """Round float32 values to the nearest bfloat16 (ties to even) and return them as float32.

    faiss flat is fp32-only; for the bf16 configurations the oracle consumes the SAME bf16 values
    upcast to fp32 (SURVEY.md §8c "bf16 parity definition")."""
    a = _f32(a)
    u = a.view(np.uint32).astype(np.uint64)
    rounded = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    out = rounded.astype(np.uint32).view(np.float32).reshape(a.shape)
    nan = np.isnan(a)
    if nan.any():
        out = out.copy()
        out[nan] = np.nan
    return out


def f32_to_bf16_bits(a) -> np.ndarray:
    """uint16 bit patterns of the bf16 rounding of a float32 array."""
    return (to_bf16_f32(a).view(np.uint32) >> 16).astype(np.uint16)


def scores(x, q, metric=IP, scorer=CANONICAL) -> np.ndarray:
    x, q = _f32(x), _f32(q)
    n, d = x.shape
    nq = q.shape[0]
    out = np.empty((nq, n), dtype=np.float32)
    lib().orc_scores(_p(x, ctypes.c_float), n, d, _p(q, ctypes.c_float), nq, metric, scorer, _p(out, ctypes.c_float))
    return out


def knn(x, q, k, metric=IP, scorer=CANONICAL):
    """IndexFlat{IP,L2}.search(q, k) restated: returns (D[nq,k] float32, I[nq,k] int64)."""
    x, q = _f32(x), _f32(q)
    n, d = x.shape
    nq = q.shape[0]
    assert q.shape[1] == d
    D = np.empty((nq, k), dtype=np.float32)
    I = np.empty((nq, k), dtype=np.int64)
    rc = lib().orc_knn(_p(x, ctypes.c_float), n, d, _p(q, ctypes.c_float), nq, k, metric, scorer,
                       _p(D, ctypes.c_float), _p(I, ctypes.c_int64))
    if rc != 0:
        raise ValueError("orc_knn failed")
    return D, I


def knn_blocked(x, q, k, metric=IP):
    """Query-blocked fp32 FMA search with the same heap code (faiss BLAS-path analogue): the timed CPU baseline."""
    x, q = _f32(x), _f32(q)
    n, d = x.shape
    nq = q.shape[0]
    D = np.empty((nq, k), dtype=np.float32)
    I = np.empty((nq, k), dtype=np.int64)
    rc = lib().orc_knn_blocked(_p(x, ctypes.c_float), n, d, _p(q, ctypes.c_float), nq, k, metric,
                               _p(D, ctypes.c_float), _p(I, ctypes.c_int64))
    if rc != 0:
        raise ValueError("orc_knn_blocked failed")
    return D, I


def knn_tiled(x, q, k, metric=IP, sb: int = 0, native: bool = True):
    """Cache-tiled fp32 FMA search (orc_knn_tiled), by default from the -march=native build: the timed CPU arm."""
    x, q = _f32(x), _f32(q)
    n, d = x.shape
    nq = q.shape[0]
    D = np.empty((nq, k), dtype=np.float32)
    I = np.empty((nq, k), dtype=np.int64)
    L = native_lib() if native else lib()
    if not hasattr(L.orc_knn_tiled, "argtypes") or L.orc_knn_tiled.argtypes is None:
        f32p, i64p = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int64)
        L.orc_knn_tiled.restype = ctypes.c_int
        L.orc_knn_tiled.argtypes = [f32p, ctypes.c_int64, ctypes.c_int, f32p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, f32p, i64p]
    rc = L.orc_knn_tiled(_p(x, ctypes.c_float), n, d, _p(q, ctypes.c_float), nq, k, metric, sb, _p(D, ctypes.c_float), _p(I, ctypes.c_int64))
    if rc != 0:
        raise ValueError("orc_knn_tiled failed")
    return D, I


def knn_sgemm(x, q, k, metric=IP, q_block: int = 2048, x_block: int = 65536):
    """Second labelled CPU arm: numpy (OpenBLAS) sgemm over (query block x corpus block) + argpartition + merge — the cache
    behaviour of faiss's BLAS path with numpy's selection instead of faiss's heap (top-k SET is the same; ties / order within
    equal scores are numpy's). IP only needs the products; L2 adds the norms like faiss (||q||^2 + ||x||^2 - 2 q.x)."""
    x, q = _f32(x), _f32(q)
    n, d = x.shape
    nq = q.shape[0]
    kk = min(k, n)
    D = np.full((nq, k), -np.finfo(np.float32).max if metric == IP else np.finfo(np.float32).max, dtype=np.float32)
    I = np.full((nq, k), -1, dtype=np.int64)
    xn = (x * x).sum(axis=1) if metric == L2 else None
    for q0 in range(0, nq, q_block):
        qb = q[q0:q0 + q_block]
        qn = (qb * qb).sum(axis=1) if metric == L2 else None
        best_s, best_i = None, None
        for x0 in range(0, n, x_block):
            xb = x[x0:x0 + x_block]
            s = qb @ xb.T
            if metric == L2:
                s = np.maximum(qn[:, None] + xn[None, x0:x0 + x_block] - 2 * s, 0)
                key = s
            else:
                key = -s
            m = min(kk, xb.shape[0])
            part = np.argpartition(key, m - 1, axis=1)[:, :m]
            ps = np.take_along_axis(s, part, axis=1)
            pi = part + x0
            if best_s is None:
                best_s, best_i = ps, pi
            else:
                cs, ci = np.concatenate([best_s, ps], axis=1), np.concatenate([best_i, pi], axis=1)
                ck = cs if metric == L2 else -cs
                sel = np.argpartition(ck, kk - 1, axis=1)[:, :kk]
                best_s, best_i = np.take_along_axis(cs, sel, axis=1), np.take_along_axis(ci, sel, axis=1)
        order = np.argsort(best_s if metric == L2 else -best_s, axis=1, kind="stable")
        D[q0:q0 + len(qb), :best_s.shape[1]] = np.take_along_axis(best_s, order, axis=1)
        I[q0:q0 + len(qb), :best_s.shape[1]] = np.take_along_axis(best_i, order, axis=1)
    return D, I


def cpu_budget() -> dict:
    """Host cores this process may really use: the affinity mask, capped by the cgroup CPU quota when the container has one
    (a container that SEES 128 cores but is allowed 16 CPU-seconds per second only thrashes with 128 threads)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        aff = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                per = float(f.read())
            if q > 0:
                quota = q / per
        except Exception:
            quota = None
    use = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    load = None
    try:
        load = os.getloadavg()[0]
    except Exception:
        pass
    return {"affinity": aff, "cgroup_quota_cpus": quota, "threads": use, "loadavg_1m": load}


def use_all_cores_native() -> int:
    n = cpu_budget()["threads"]
    native_lib().orc_set_num_threads(n)
    return int(native_lib().orc_num_threads())


def knn_subset(x, q, k, ids, metric=IP, scorer=CANONICAL):
    """FaissVS.__call__ with ids (faiss_vs.py:57-72): temp index over x[ids], search, remap.
    The reference's -1 wrap-around bug when k > len(ids) is NOT reproduced: -1 stays -1."""
    ids = np.asarray(ids, dtype=np.int64)
    D, sub = knn(_f32(x)[ids], q, k, metric, scorer)
    I = np.where(sub >= 0, ids[np.clip(sub, 0, max(len(ids) - 1, 0))] if len(ids) else -1, -1)
    return D, I.astype(np.int64)


def knn_window_rule(S: np.ndarray, k: int, metric=IP):
    """Closed form of what the faiss heap retains, derived in DESIGN.md §Ties, written with numpy from
    a dense score matrix S[nq,n]. Independent of the heap code in faiss_flat.c; the two must agree."""
    nq, n = S.shape
    D = np.full((nq, k), -np.finfo(np.float32).max if metric == IP else np.finfo(np.float32).max, dtype=np.float32)
    I = np.full((nq, k), -1, dtype=np.int64)
    for qi in range(nq):
        s = S[qi]
        ids = np.arange(n)
        key = -s.astype(np.float64) if metric == IP else s.astype(np.float64)
        if n <= k:
            keep = ids
        else:
            order = np.lexsort((ids, key))  # best first, ties by id asc
            v = key[order[k - 1]]
            better = ids[key < v]
            ties = ids[key == v]  # ascending id
            r = k - len(better)
            if metric == L2 or k == 1:
                kept_ties = ties[:r]
            else:
                sset = np.sort(np.concatenate([better, ties]))[:k]  # first k (by id) of {score >= v}
                t = int(np.isin(ties, sset).sum())
                kept_ties = ties[t - r:t]
            keep = np.concatenate([better, kept_ties])
        kk = key[keep]
        if metric == IP and k > 1:
            o = np.lexsort((-keep, kk))  # score desc, id desc
        else:
            o = np.lexsort((keep, kk))  # best first, id asc
        keep = keep[o]
        m = len(keep)
        D[qi, :m] = s[keep]
        I[qi, :m] = keep
    return D, I


def threshold_pairs(x, thr: float, cap: int | None = None):
    x = _f32(x)
    n, d = x.shape
    cap = int(cap if cap is not None else max(n * (n - 1) // 2, 1))
    oi = np.empty(cap, dtype=np.int64)
    oj = np.empty(cap, dtype=np.int64)
    cnt = lib().orc_threshold_pairs(_p(x, ctypes.c_float), n, d, float(thr), _p(oi, ctypes.c_int64),
                                    _p(oj, ctypes.c_int64), cap)
    m = min(cnt, cap)
    return oi[:m].copy(), oj[:m].copy(), int(cnt)


def connected_components(n: int, pi, pj) -> np.ndarray:
    """labels[i] = smallest row id in i's component (sem_dedup.py:58-84 computes the same partition
    by DFS over text values)."""
    parent = np.arange(n, dtype=np.int64)

    def find(a):
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a

    for a, b in zip(np.asarray(pi).tolist(), np.asarray(pj).tolist()):
        ra, rb = find(a), find(b)
        if ra != rb:
            if ra < rb:
                parent[rb] = ra
            else:
                parent[ra] = rb
    return np.array([find(i) for i in range(n)], dtype=np.int64)


def mt19937(seed: int, count: int) -> np.ndarray:
    out = np.empty(count, dtype=np.uint32)
    lib().orc_mt_fill(seed & 0xFFFFFFFF, _p(out, ctypes.c_uint32), count)
    return out


def rand_perm(n: int, seed: int) -> np.ndarray:
    out = np.empty(n, dtype=np.int32)
    lib().orc_rand_perm(_p(out, ctypes.c_int32), n, seed)
    return out


def kmeans(x, k: int, niter: int = 20, seed: int = 1234, scorer=CANONICAL, full_lloyd: bool = False):
    """faiss.Kmeans(d,k,niter=niter).train(x); index.search(x,1) -> (assign[n], centroids[k,d], obj[niter])."""
    x = _f32(x)
    n, d = x.shape
    assign = np.empty(n, dtype=np.int64)
    cent = np.zeros((k, d), dtype=np.float32)
    obj = np.zeros(max(niter, 1), dtype=np.float32)
    rc = lib().orc_kmeans(_p(x, ctypes.c_float), n, d, k, niter, seed, scorer, int(full_lloyd),
                          _p(assign, ctypes.c_int64), _p(cent, ctypes.c_float), _p(obj, ctypes.c_float))
    if rc != 0:
        raise ValueError(f"Number of training points ({n}) should be at least as large as number of clusters ({k})")
    return assign, cent, obj[:niter]


def compute_centroids(x, assign, k: int):
    x = _f32(x)
    n, d = x.shape
    assign = np.ascontiguousarray(assign, dtype=np.int64)
    h = np.zeros(k, dtype=np.float32)
    c = np.zeros((k, d), dtype=np.float32)
    lib().orc_compute_centroids(d, k, n, _p(x, ctypes.c_float), _p(assign, ctypes.c_int64), _p(h, ctypes.c_float),
                                _p(c, ctypes.c_float))
    return c, h


def split_clusters(centroids, hassign, n: int):
    c = _f32(centroids).copy()
    h = _f32(hassign).copy()
    k, d = c.shape
    ns = lib().orc_split_clusters(d, k, n, _p(h, ctypes.c_float), _p(c, ctypes.c_float))
    return c, h, int(ns)
