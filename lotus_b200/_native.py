"""ctypes binding of libb2lotus.so (include/lotus_b200.h). No CPU fallback: if the library is not built or no
B200 is visible, calls raise — they never degrade to a host implementation."""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb2lotus.so")

F32, BF16, F16 = 0, 1, 2
METRIC_IP, METRIC_L2 = 0, 1
OK, EINVAL, ENODEV, ECUDA, ENOMEM, ERANGE = 0, -1, -2, -3, -4, -5

# every symbol include/lotus_b200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "b2_abi_version", "b2_last_error", "b2_device_count", "b2_max_k", "b2_index_create", "b2_index_free",
    "b2_index_ntotal", "b2_index_dim", "b2_index_dtype", "b2_index_metric", "b2_index_device", "b2_index_data_dev",
    "b2_index_search", "b2_index_search_dev", "b2_merge_topk_dev", "b2_index_search_packed_dev", "b2_merge_topk_packed_dev", "b2_index_search_stage1_dev", "b2_index_search_stage2_packed_dev", "b2_index_gather", "b2_threshold_pairs",
    "b2_connected_components", "b2_kmeans", "b2_kmeans_assign", "b2_kmeans_accumulate", "b2_kmeans_assign_dev", "b2_kmeans_accumulate_dev", "b2_stats", "b2_stats_reset", "b2_last_filter_ms", "b2_host_f32_to_bf16", "b2_host_bf16_to_f32", "b2_debug_filter_plan",
]


class NativeError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libb2lotus error {code}: {msg}")
        self.code = code
        self.msg = msg


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m lotus_b200.build` "
            "(lotus_b200 has no CPU fallback and refuses to run without its CUDA library)")
    L = ctypes.CDLL(LIB_PATH)
    c = ctypes
    vp, i32, i64, f32 = c.c_void_p, c.c_int32, c.c_int64, c.c_float
    L.b2_abi_version.restype = c.c_int
    L.b2_last_error.restype = c.c_char_p
    L.b2_device_count.restype = c.c_int
    L.b2_max_k.restype = c.c_int
    L.b2_index_create.restype = c.c_int
    L.b2_index_create.argtypes = [vp, i64, i32, i32, i32, i32, i32, c.POINTER(vp)]
    L.b2_index_free.restype = None
    L.b2_index_free.argtypes = [vp]
    for name, rt in [("b2_index_ntotal", i64), ("b2_index_dim", i32), ("b2_index_dtype", i32),
                     ("b2_index_metric", i32), ("b2_index_device", i32), ("b2_index_data_dev", vp),
                     ("b2_last_filter_ms", f32)]:
        getattr(L, name).restype = rt
        getattr(L, name).argtypes = [vp]
    L.b2_index_search.restype = c.c_int
    L.b2_index_search.argtypes = [vp, vp, i64, i32, i32, vp, i64, vp, vp]
    L.b2_index_search_dev.restype = c.c_int
    L.b2_index_search_dev.argtypes = [vp, vp, i64, i32, i32, vp, i64, i64, vp, vp, vp]
    L.b2_merge_topk_dev.restype = c.c_int
    L.b2_merge_topk_dev.argtypes = [vp, vp, i32, i64, i32, i32, i32, vp, vp, vp]
    L.b2_index_search_packed_dev.restype = c.c_int
    L.b2_index_search_packed_dev.argtypes = [vp, vp, i64, i32, i32, vp, vp]
    L.b2_merge_topk_packed_dev.restype = c.c_int
    L.b2_merge_topk_packed_dev.argtypes = [vp, vp, i32, i64, i32, i32, i32, vp, vp, vp]
    L.b2_index_search_stage1_dev.restype = c.c_int
    L.b2_index_search_stage1_dev.argtypes = [vp, vp, i64, i32, i32, i32, vp, vp]
    L.b2_index_search_stage2_packed_dev.restype = c.c_int
    L.b2_index_search_stage2_packed_dev.argtypes = [vp, vp, vp, vp]
    L.b2_index_gather.restype = c.c_int
    L.b2_index_gather.argtypes = [vp, vp, i64, vp, i32]
    L.b2_threshold_pairs.restype = c.c_int
    L.b2_threshold_pairs.argtypes = [vp, f32, i32, i32, vp, vp, i64, c.POINTER(i64)]
    L.b2_connected_components.restype = c.c_int
    L.b2_connected_components.argtypes = [i64, vp, vp, i64, i32, vp]
    L.b2_kmeans.restype = c.c_int
    L.b2_kmeans.argtypes = [vp, vp, i64, i32, i32, i64, i32, vp, vp, vp]
    L.b2_kmeans_assign.restype = c.c_int
    L.b2_kmeans_assign.argtypes = [vp, vp, i64, vp, i32, vp, vp]
    L.b2_kmeans_accumulate.restype = c.c_int
    L.b2_kmeans_accumulate.argtypes = [vp, vp, i64, vp, i32, vp, vp]
    L.b2_kmeans_assign_dev.restype = c.c_int
    L.b2_kmeans_assign_dev.argtypes = [vp, vp, i64, vp, i32, vp, vp, vp]
    L.b2_kmeans_accumulate_dev.restype = c.c_int
    L.b2_kmeans_accumulate_dev.argtypes = [vp, vp, i64, vp, i32, vp, vp, vp, vp, vp]
    L.b2_host_f32_to_bf16.restype = c.c_int
    L.b2_host_f32_to_bf16.argtypes = [vp, i64, vp, c.POINTER(i32)]
    L.b2_host_bf16_to_f32.restype = c.c_int
    L.b2_host_bf16_to_f32.argtypes = [vp, i64, vp]
    L.b2_debug_filter_plan.restype = c.c_int
    L.b2_debug_filter_plan.argtypes = [i64, i64, i32, i32, c.POINTER(i32), c.POINTER(i32), c.POINTER(i32), c.POINTER(i32)]
    L.b2_stats.restype = c.c_int
    L.b2_stats.argtypes = [c.POINTER(i64), i32]
    L.b2_stats_reset.restype = None
    if L.b2_abi_version() != 1:
        raise RuntimeError("libb2lotus.so ABI version mismatch; rebuild with `python -m lotus_b200.build --force`")
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        raise NativeError(rc, lib().b2_last_error().decode("utf-8", "replace"))


def device_count() -> int:
    return int(lib().b2_device_count())


def require_device() -> None:
    if device_count() == 0:
        raise RuntimeError("lotus_b200 needs a B200 (sm_100) GPU; none is visible and there is no CPU fallback")


def filter_plan(nq: int, n: int, k: int, num_sms: int = 148) -> dict:
    """The filter kernel's schedule for a shape (host logic only, no device needed)."""
    kp, ns, uw, two = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    check(lib().b2_debug_filter_plan(nq, n, k, num_sms, ctypes.byref(kp), ctypes.byref(ns), ctypes.byref(uw), ctypes.byref(two)))
    return {"kp": kp.value, "n_splits": ns.value, "units_whole": uw.value, "two_cta": bool(two.value)}


def stats() -> dict:
    buf = (ctypes.c_int64 * 8)()
    lib().b2_stats(buf, 8)
    return {"launches": buf[0], "queries": buf[1], "fallback_queries": buf[2], "filter_launches": buf[3],
            "rescored_rows": buf[4], "second_level_queries": buf[5]}


def stats_reset() -> None:
    lib().b2_stats_reset()


# ---- bf16 helpers (numpy has no bfloat16: bit patterns travel as uint16) ------------------------------------------
def f32_to_bf16_checked(a: np.ndarray, out: "np.ndarray | None" = None) -> tuple[np.ndarray, bool]:
    """Round-to-nearest-even float32 -> bfloat16 bit patterns (uint16; NaN stays a quiet NaN) plus whether every value
    was already bfloat16-representable. Host marshalling done by the library's threaded helper (no device work). `out`: a
    C-contiguous uint16 array of the same shape to write into (callers that convert a batch per call keep one: a fresh 150 MB
    array costs more in page faults than the conversion itself)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    if out is None or out.shape != a.shape or out.dtype != np.uint16 or not out.flags.c_contiguous:
        out = np.empty(a.shape, dtype=np.uint16)
    exact = ctypes.c_int32(0)
    check(lib().b2_host_f32_to_bf16(_ptr(a), a.size, _ptr(out), ctypes.byref(exact)))
    return out, bool(exact.value)


def f32_to_bf16_bits(a: np.ndarray) -> np.ndarray:
    """Round-to-nearest-even float32 -> bfloat16 bit patterns (uint16)."""
    return f32_to_bf16_checked(a)[0]


def bf16_bits_to_f32(b: np.ndarray) -> np.ndarray:
    b = np.ascontiguousarray(b, dtype=np.uint16)
    if b.size < (1 << 18):
        return (b.astype(np.uint32) << 16).view(np.float32).reshape(b.shape)
    out = np.empty(b.shape, dtype=np.float32)
    check(lib().b2_host_bf16_to_f32(_ptr(b), b.size, _ptr(out)))
    return out


# ---- fp16 helpers (numpy's float16 is IEEE binary16: RNE conversions, so plain numpy does the marshalling) ----------------
F16_MAX = 65504.0


def f32_to_f16_bits(a: np.ndarray) -> np.ndarray:
    """Round-to-nearest-even float32 -> float16 bit patterns (uint16). Values beyond fp16's range become inf."""
    with np.errstate(over="ignore"):
        return np.ascontiguousarray(a, dtype=np.float32).astype(np.float16).view(np.uint16)


def f16_bits_to_f32(b: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(b, dtype=np.uint16).view(np.float16).astype(np.float32)


def bits_to_f32(a: np.ndarray, code: int) -> np.ndarray:
    """float32 values of a matrix in the library's element type `code` (2-byte types travel as uint16 bit patterns)."""
    if code == BF16:
        return bf16_bits_to_f32(a)
    if code == F16:
        return f16_bits_to_f32(a)
    return a


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


class Index:
    """Owning wrapper of a b2_index handle."""

    def __init__(self, x, dtype: int, metric: int = METRIC_IP, device: int = 0, on_device_ptr: Optional[int] = None,
                 n: Optional[int] = None, d: Optional[int] = None):
        L = lib()
        self._h = ctypes.c_void_p()
        if on_device_ptr is not None:
            assert n is not None and d is not None
            check(L.b2_index_create(ctypes.c_void_p(on_device_ptr), n, d, dtype, metric, device, 1, ctypes.byref(self._h)))
        else:
            x = np.ascontiguousarray(x)
            want = np.float32 if dtype == F32 else np.uint16
            if x.dtype != want:
                raise TypeError(f"matrix must be {want} for dtype {dtype}, got {x.dtype}")
            if x.ndim != 2:
                raise ValueError("matrix must be 2-D")
            n, d = x.shape
            check(L.b2_index_create(_ptr(x) if n else None, n, d, dtype, metric, device, 0, ctypes.byref(self._h)))
        self.n, self.d, self.dtype, self.metric, self.device = int(n), int(d), dtype, metric, device

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().b2_index_free(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    @property
    def data_ptr(self) -> int:
        return int(lib().b2_index_data_dev(self._h) or 0)

    def search(self, q: np.ndarray, k: int, q_dtype: int = F32, ids: Optional[np.ndarray] = None):
        """Host buffers in, host buffers out: (scores[nq,k] float32, idx[nq,k] int64)."""
        q = np.ascontiguousarray(q)
        nq = q.shape[0]
        if nq and q.shape[1] != self.d:
            raise ValueError(f"query dimension {q.shape[1]} != index dimension {self.d}")
        D = np.empty((nq, k), dtype=np.float32)
        I = np.empty((nq, k), dtype=np.int64)
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.int64)
        check(lib().b2_index_search(self._h, _ptr(q) if nq else None, nq, q_dtype, k, _ptr(ids_a),
                                    0 if ids_a is None else len(ids_a), _ptr(D), _ptr(I)))
        return D, I

    def search_dev(self, q_ptr: int, nq: int, k: int, q_dtype: int, out_scores_ptr: int, out_idx_ptr: int,
                   id_offset: int = 0, ids_ptr: Optional[int] = None, n_ids: int = 0, stream: int = 0) -> None:
        check(lib().b2_index_search_dev(self._h, ctypes.c_void_p(q_ptr), nq, q_dtype, k,
                                        ctypes.c_void_p(ids_ptr) if ids_ptr else None, n_ids, id_offset,
                                        ctypes.c_void_p(out_scores_ptr), ctypes.c_void_p(out_idx_ptr),
                                        ctypes.c_void_p(stream) if stream else None))

    def search_packed_dev(self, q_ptr: int, nq: int, k: int, q_dtype: int, out_packed_ptr: int, stream: int = 0) -> None:
        """Whole-index search, result as one uint64 per entry (float32 score bits << 32 | local row id, 0xffffffff = none)."""
        check(lib().b2_index_search_packed_dev(self._h, ctypes.c_void_p(q_ptr), nq, q_dtype, k, ctypes.c_void_p(out_packed_ptr),
                                               ctypes.c_void_p(stream) if stream else None))

    def search_stage1_dev(self, q_ptr: int, nq: int, k: int, q_dtype: int, j: int, lower_ptr: int, stream: int = 0) -> None:
        check(lib().b2_index_search_stage1_dev(self._h, ctypes.c_void_p(q_ptr), nq, q_dtype, k, j, ctypes.c_void_p(lower_ptr),
                                               ctypes.c_void_p(stream) if stream else None))

    def search_stage2_packed_dev(self, hint_ptr: int, out_packed_ptr: int, stream: int = 0) -> None:
        check(lib().b2_index_search_stage2_packed_dev(self._h, ctypes.c_void_p(hint_ptr), ctypes.c_void_p(out_packed_ptr),
                                                      ctypes.c_void_p(stream) if stream else None))

    def gather(self, ids) -> np.ndarray:
        """Rows in the index's element type (uint16 bit patterns for BF16 / F16)."""
        ids = np.ascontiguousarray(ids, dtype=np.int64)
        out = np.empty((len(ids), self.d), dtype=np.float32 if self.dtype == F32 else np.uint16)
        check(lib().b2_index_gather(self._h, _ptr(ids), len(ids), _ptr(out), 0))
        return out

    def last_filter_ms(self) -> float:
        return float(lib().b2_last_filter_ms(self._h))

    def threshold_pairs(self, thr: float, cap: int = 1 << 24, part: int = 0, nparts: int = 1):
        oi = np.empty(cap, dtype=np.int64)
        oj = np.empty(cap, dtype=np.int64)
        cnt = ctypes.c_int64(0)
        rc = lib().b2_threshold_pairs(self._h, float(thr), part, nparts, _ptr(oi), _ptr(oj), cap, ctypes.byref(cnt))
        if rc == ERANGE and cnt.value > cap:
            return self.threshold_pairs(thr, cap=int(cnt.value), part=part, nparts=nparts)
        check(rc)
        m = int(cnt.value)
        return oi[:m].copy(), oj[:m].copy()

    def kmeans(self, k: int, niter: int = 20, seed: int = 1234, ids=None, full_lloyd: bool = False):
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.int64)
        m = self.n if ids_a is None else len(ids_a)
        assign = np.empty(m, dtype=np.int64)
        cent = np.empty((k, self.d), dtype=np.float32)
        obj = np.zeros(max(niter, 1), dtype=np.float32)
        check(lib().b2_kmeans(self._h, _ptr(ids_a), m, k, niter, seed, int(full_lloyd), _ptr(assign), _ptr(cent), _ptr(obj)))
        return assign, cent, obj[:niter]

    def kmeans_assign(self, centroids: np.ndarray, ids=None):
        c = np.ascontiguousarray(centroids, dtype=np.float32)
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.int64)
        m = self.n if ids_a is None else len(ids_a)
        assign = np.empty(m, dtype=np.int64)
        dist = np.empty(m, dtype=np.float32)
        check(lib().b2_kmeans_assign(self._h, _ptr(ids_a), m, _ptr(c), c.shape[0], _ptr(assign), _ptr(dist)))
        return assign, dist


def merge_topk_packed_dev(packed_ptr: int, shard_offsets, g: int, nq: int, k: int, metric: int, device: int,
                          out_scores_ptr: int, out_idx_ptr: int, stream: int = 0) -> None:
    offs = np.ascontiguousarray(shard_offsets, dtype=np.int64)
    assert len(offs) == g
    check(lib().b2_merge_topk_packed_dev(ctypes.c_void_p(packed_ptr), _ptr(offs), g, nq, k, metric, device,
                                         ctypes.c_void_p(out_scores_ptr), ctypes.c_void_p(out_idx_ptr),
                                         ctypes.c_void_p(stream) if stream else None))


def _index_kmeans_assign_dev(self, centroids_ptr: int, k: int, assign_ptr: int, dist_ptr: int = 0, ids_ptr: int = 0, m: int = 0,
                             stream: int = 0) -> None:
    """DEVICE buffers: assign[m] int64 (and dist[m] float32 when dist_ptr) against centroids[k,d] float32."""
    check(lib().b2_kmeans_assign_dev(self._h, ctypes.c_void_p(ids_ptr) if ids_ptr else None, m, ctypes.c_void_p(centroids_ptr), k,
                                     ctypes.c_void_p(assign_ptr), ctypes.c_void_p(dist_ptr) if dist_ptr else None,
                                     ctypes.c_void_p(stream) if stream else None))


def _index_kmeans_accumulate_dev(self, assign_ptr: int, k: int, sums_ptr: int, counts_ptr: int, centroids_ptr: int = 0, obj_ptr: int = 0,
                                 ids_ptr: int = 0, m: int = 0, stream: int = 0) -> None:
    """DEVICE buffers: per-shard point-order sums[k,d] + counts[k] (float32); *obj += sum of squared distances (float64)."""
    check(lib().b2_kmeans_accumulate_dev(self._h, ctypes.c_void_p(ids_ptr) if ids_ptr else None, m, ctypes.c_void_p(assign_ptr), k,
                                         ctypes.c_void_p(centroids_ptr) if centroids_ptr else None, ctypes.c_void_p(sums_ptr),
                                         ctypes.c_void_p(counts_ptr), ctypes.c_void_p(obj_ptr) if obj_ptr else None,
                                         ctypes.c_void_p(stream) if stream else None))


def pair_owner(i, nparts: int):
    """Rank that owns the pairs (i, j > i) in `threshold_pairs(part=, nparts=)`: 128-row query tiles are dealt to the ranks in
    groups of one tile per SM (148 on B200; B2_PAIR_GROUP overrides) — mirrors launch_pair_filter in knn_filter_sm100.cu."""
    group = int(os.environ.get("B2_PAIR_GROUP", "0")) or 148
    tile = np.asarray(i, dtype=np.int64) // 128
    if int(os.environ.get("B2_PAIR_2CTA", "1")):  # CTA pairs (default): the unit is two consecutive query tiles, one unit per pair of SMs
        return ((tile // 2) // max(1, group // 2)) % nparts
    return (tile // group) % nparts


def _index_kmeans_accumulate(self, assign, k: int, ids=None):
    """Per-shard centroid sums [k,d] (point order, fp32, not normalised) and counts [k] for multi-GPU Lloyd."""
    a = np.ascontiguousarray(assign, dtype=np.int64)
    ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.int64)
    sums = np.empty((k, self.d), dtype=np.float32)
    counts = np.empty(k, dtype=np.float32)
    check(lib().b2_kmeans_accumulate(self._h, _ptr(ids_a), len(a), _ptr(a), k, _ptr(sums), _ptr(counts)))
    return sums, counts


Index.kmeans_accumulate = _index_kmeans_accumulate
Index.kmeans_assign_dev = _index_kmeans_assign_dev
Index.kmeans_accumulate_dev = _index_kmeans_accumulate_dev


def connected_components(n: int, pi: np.ndarray, pj: np.ndarray, device: int = 0) -> np.ndarray:
    pi = np.ascontiguousarray(pi, dtype=np.int64)
    pj = np.ascontiguousarray(pj, dtype=np.int64)
    labels = np.empty(n, dtype=np.int64)
    check(lib().b2_connected_components(n, _ptr(pi), _ptr(pj), len(pi), device, _ptr(labels)))
    return labels


def merge_topk_dev(scores_ptr: int, idx_ptr: int, g: int, nq: int, k: int, metric: int, device: int,
                   out_scores_ptr: int, out_idx_ptr: int, stream: int = 0) -> None:
    check(lib().b2_merge_topk_dev(ctypes.c_void_p(scores_ptr), ctypes.c_void_p(idx_ptr), g, nq, k, metric, device,
                                  ctypes.c_void_p(out_scores_ptr), ctypes.c_void_p(out_idx_ptr),
                                  ctypes.c_void_p(stream) if stream else None))
