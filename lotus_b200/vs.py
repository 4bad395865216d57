"""Vector-store boundary: the `VS` ABC of the reference (lotus/vector_store/vs.py:10-58) and `B200VS`, the
drop-in replacement of `FaissVS` (lotus/vector_store/faiss_vs.py:13-77) backed by libb2lotus.so.

    lotus.settings.configure(rm=rm, vs=B200VS())          # where the reference says vs=FaissVS()

There is no CPU path: without the CUDA library / a B200 every method that computes raises.
"""
from __future__ import annotations

import os
from abc import ABC, abstractmethod
from collections import OrderedDict
from typing import Any

import numpy as np

from . import _native as nv
from . import faiss_io
from .types import RMOutput

try:  # when the real package is importable, plug into ITS class hierarchy so isinstance checks pass
    from lotus.vector_store.vs import VS as _RefVS  # type: ignore
    from lotus.types import RMOutput as _RefRMOutput  # type: ignore
    RMOutput = _RefRMOutput  # noqa: F811
except Exception:  # lotus (litellm, faiss, ...) is not importable in this image: mirror the ABC
    _RefVS = None

METRIC_INNER_PRODUCT = faiss_io.METRIC_INNER_PRODUCT  # == faiss.METRIC_INNER_PRODUCT
METRIC_L2 = faiss_io.METRIC_L2  # == faiss.METRIC_L2

if _RefVS is not None:
    VS = _RefVS
else:

    class VS(ABC):  # type: ignore[no-redef]
        """Abstract class for vector stores (lotus/vector_store/vs.py:10-58)."""

        def __init__(self) -> None:
            self.index_dir: str | None = None

        @abstractmethod
        def index(self, docs: Any, embeddings: Any, index_dir: str, **kwargs: Any):
            ...

        @abstractmethod
        def load_index(self, index_dir: str):
            ...

        @abstractmethod
        def __call__(self, query_vectors: Any, K: int, ids: list[int] | None = None, **kwargs: Any) -> RMOutput:
            ...

        @abstractmethod
        def get_vectors_from_index(self, index_dir: str, ids: list[int]) -> Any:
            ...


def _cuda_tensor(a: Any):
    """The tensor itself when `a` is a torch CUDA tensor (device hand-off, SURVEY §8f-2), else None."""
    try:
        import torch
        if isinstance(a, torch.Tensor) and a.is_cuda:
            return a
    except ImportError:  # pragma: no cover
        pass
    return None


class BF16Backed(np.ndarray):
    """float32 matrix handed out by `B200VS.get_vectors_from_index` for bf16 indexes. It is a plain float32 array to every
    caller; the name only records where it came from. (Round 1 carried the bf16 bit patterns along as an attribute; an
    in-place edit such as `q /= norm` left them stale. `B200VS.__call__` now re-derives the 2-byte form from the VALUES —
    see `_to_host_matrix(exact_bf16_ok=True)` — so nothing can go stale.)"""

    @staticmethod
    def wrap(f32: np.ndarray, bits: "np.ndarray | None" = None) -> "BF16Backed":
        return np.ascontiguousarray(f32, dtype=np.float32).view(BF16Backed)


def _to_host_matrix(a: Any, want_bf16: bool, exact_bf16_ok: bool = False, scratch: "dict | None" = None, want_f16: bool = False,
                    exact_f16_ok: bool = False):
    """-> (array for the C-ABI, native dtype code, float32 view of the stored values).
    exact_bf16_ok: when every float32 value is bfloat16-representable (e.g. vectors fetched from a bf16 index,
    sem_sim_join.py:112-118 -> :130-134) ship the exact 2-byte patterns instead: half the H2D bytes and the exact-operand
    error bound in the certificate. Decided from the values themselves on every call (one threaded host pass).
    want_f16 / exact_f16_ok: the same for fp16 (IEEE binary16, rounded to nearest even by numpy); want_f16 rounds, and a value
    beyond fp16's finite range raises ValueError."""
    try:
        import torch
        if isinstance(a, torch.Tensor):
            t = a.detach()
            if t.dtype == torch.float16 and (want_f16 or exact_f16_ok):
                bits = t.contiguous().cpu().view(torch.int16).numpy().view(np.uint16)
                return bits, nv.F16, nv.f16_bits_to_f32(bits)
            if t.dtype == torch.bfloat16 or want_bf16:
                bits = t.to(torch.bfloat16).contiguous().cpu().view(torch.int16).numpy().view(np.uint16)
                return bits, nv.BF16, nv.bf16_bits_to_f32(bits)
            a = t.to(torch.float32).contiguous().cpu().numpy()
    except ImportError:  # pragma: no cover
        pass
    f = np.ascontiguousarray(np.asarray(a), dtype=np.float32)  # faiss casts whatever it is given to float32
    if f.ndim != 2:
        raise ValueError(f"embeddings must be 2-D, got shape {f.shape}")
    if want_f16:
        bits = nv.f32_to_f16_bits(f)
        _check_f16_range(bits)
        return bits, nv.F16, nv.f16_bits_to_f32(bits)
    if exact_f16_ok and f.size:
        bits = nv.f32_to_f16_bits(f)
        if np.array_equal(nv.f16_bits_to_f32(bits), f):
            return bits, nv.F16, f
    if want_bf16:
        bits = nv.f32_to_bf16_bits(f)
        return bits, nv.BF16, nv.bf16_bits_to_f32(bits)
    if exact_bf16_ok and f.size:
        buf = None
        if scratch is not None:  # one reusable staging array per store (the C call copies it to the device before returning)
            buf = scratch.get("q16")
            if buf is None or buf.size < f.size:
                buf = scratch["q16"] = np.empty(f.size, dtype=np.uint16)
            buf = buf[:f.size].reshape(f.shape)
        bits, exact = nv.f32_to_bf16_checked(f, out=buf)
        if exact:
            return bits, nv.BF16, f
    return f, nv.F32, f


def _check_f16_range(bits: np.ndarray) -> None:
    """An fp16 store holds finite values only: faiss's SQfp16 would store inf for |x| >= 65520; this store refuses."""
    if bits.size and ((bits & 0x7C00) == 0x7C00).any():
        raise ValueError("embeddings have values beyond the finite range of fp16 (|x| >= 65520, or inf / NaN); an fp16 store "
                         "(dtype='f16' or factory_string='SQfp16') cannot hold them")


class MultiDeviceIndex:
    """Row-sharded flat index over several B200s driven from ONE process (for users who do not run under torchrun; under
    torchrun use lotus_b200.distributed.ShardedIndex, whose exchange runs over NCCL/NVLink). Shard g holds the contiguous rows
    `shard_bounds(n, G, g)` on devices[g]; a search runs the G per-device C-ABI calls concurrently (ctypes releases the GIL),
    then merges the G sorted lists on the host with the same (score, shard order) rule as the k-way merge kernel.
    Same surface as `_native.Index` as far as B200VS uses it."""

    def __init__(self, host_matrix: np.ndarray, code: int, metric: int, devices: list[int]):
        from concurrent.futures import ThreadPoolExecutor
        from .distributed import shard_bounds
        self.devices = list(devices)
        self.n, self.d = host_matrix.shape
        self.dtype, self.metric, self.device = code, metric, self.devices[0]
        self.bounds = [shard_bounds(self.n, len(self.devices), g) for g in range(len(self.devices))]
        self.pool = ThreadPoolExecutor(max_workers=len(self.devices))
        self.shards = list(self.pool.map(lambda gb: nv.Index(np.ascontiguousarray(host_matrix[gb[1][0]:gb[1][1]]), code, metric, gb[0]),
                                         zip(self.devices, self.bounds)))
        self._host = host_matrix  # kept for the operators that need the whole matrix on one device (dedup, k-means)
        self._replica: nv.Index | None = None

    def search(self, q: np.ndarray, k: int, q_dtype: int = nv.F32, ids: np.ndarray | None = None):
        def one(g):
            lo, hi = self.bounds[g]
            if ids is None:
                D, I = self.shards[g].search(q, k, q_dtype)
            else:
                mine = ids[(ids >= lo) & (ids < hi)] - lo
                if len(mine) == 0:
                    pad = np.finfo(np.float32).max if self.metric == nv.METRIC_L2 else -np.finfo(np.float32).max
                    return np.full((len(q), k), pad, np.float32), np.full((len(q), k), -1, np.int64)
                D, I = self.shards[g].search(q, k, q_dtype, ids=np.ascontiguousarray(mine))
            return D, np.where(I >= 0, I + lo, -1)
        if ids is not None and len(ids) and (ids.min() < 0 or ids.max() >= self.n):
            raise nv.NativeError(nv.ERANGE, f"ids contains a position outside [0, {self.n})")
        parts = list(self.pool.map(one, range(len(self.shards))))
        return merge_shard_lists([p[0] for p in parts], [p[1] for p in parts], self.metric)

    def gather(self, ids) -> np.ndarray:
        ids = np.asarray(ids, dtype=np.int64)
        if len(ids) and (ids.min() < 0 or ids.max() >= self.n):
            raise nv.NativeError(nv.ERANGE, f"ids contains a position outside [0, {self.n})")
        out = np.empty((len(ids), self.d), dtype=np.float32 if self.dtype == nv.F32 else np.uint16)  # BF16 / F16: bit patterns
        for g, (lo, hi) in enumerate(self.bounds):
            m = (ids >= lo) & (ids < hi)
            if m.any():
                out[m] = self.shards[g].gather(ids[m] - lo)
        return out

    def _whole(self) -> "nv.Index":
        if self._replica is None:  # all-pairs dedup and k-means want the whole matrix on one device
            self._replica = nv.Index(np.ascontiguousarray(self._host), self.dtype, self.metric, self.devices[0])
        return self._replica

    def threshold_pairs(self, thr: float, **kw):
        return self._whole().threshold_pairs(thr, **kw)

    def kmeans(self, k: int, **kw):
        return self._whole().kmeans(k, **kw)

    def close(self) -> None:
        for s in self.shards:
            s.close()
        if self._replica is not None:
            self._replica.close()
        self.pool.shutdown(wait=False)


def merge_shard_lists(D_parts: list, I_parts: list, metric: int):
    """Host k-way merge of per-shard (score, global id) lists [nq, k] -> [nq, k]: best first; equal scores keep each shard's
    (already faiss-ordered) list order, lower shards first for L2, higher shards first for IP — the rule of merge_topk_kernel."""
    g = len(D_parts)
    order = range(g) if metric == nv.METRIC_L2 else range(g - 1, -1, -1)
    D = np.concatenate([D_parts[i] for i in order], axis=1)
    I = np.concatenate([I_parts[i] for i in order], axis=1)
    k = D_parts[0].shape[1]
    key = np.where(I >= 0, D if metric == nv.METRIC_L2 else -D, np.inf)
    sel = np.argsort(key, axis=1, kind="stable")[:, :k]
    return np.take_along_axis(D, sel, axis=1), np.take_along_axis(I, sel, axis=1)


class B200VS(VS):
    """Flat (brute-force, exact) vector store on one B200 (or, with devices=[...], row-sharded over several from one process).

    Args mirror FaissVS(factory_string="Flat", metric=faiss.METRIC_INNER_PRODUCT) (faiss_vs.py:14).
    factory_string: "Flat", or "SQfp16" — faiss IndexScalarQuantizer(d, QT_fp16): the rows are stored rounded to fp16, fp32
    queries are scored exactly against them, and `get_vectors_from_index` returns the ORIGINAL embeddings (faiss_vs.py:38-41).
    dtype: "f32" (store what faiss would: float32), "bf16" / "f16" (round the corpus to bfloat16 / fp16 once; exact search
    over those values), or "auto" (bf16 only when handed a bf16 tensor). "SQfp16" implies "f16".
    """

    accepts_id_arrays = True  # `ids=` may be a numpy int64 array (the operators then skip building a Python list)

    def __init__(self, factory_string: str = "Flat", metric: int = METRIC_INNER_PRODUCT, dtype: str = "auto",
                 device: int = 0, cache_size: int = 4, devices: "list[int] | None" = None):
        super().__init__()
        if factory_string not in (faiss_io.FLAT, faiss_io.SQFP16):
            raise ValueError(f"B200VS implements the flat (exact) index types 'Flat' and 'SQfp16' only; factory_string={factory_string!r}")
        if metric not in (METRIC_INNER_PRODUCT, METRIC_L2):
            raise ValueError("metric must be METRIC_INNER_PRODUCT (0) or METRIC_L2 (1)")
        if dtype not in ("auto", "f32", "bf16", "f16"):
            raise ValueError("dtype must be 'auto', 'f32', 'bf16' or 'f16'")
        self.sq = factory_string == faiss_io.SQFP16
        if self.sq:
            if dtype not in ("auto", "f16"):
                raise ValueError(f"factory_string='SQfp16' stores fp16 rows; dtype={dtype!r} contradicts it")
            dtype = "f16"
        self.factory_string = factory_string
        self.metric = metric
        self.dtype = dtype
        self.devices = list(devices) if devices else None
        self.device = self.devices[0] if self.devices else device
        self.index_dir: str | None = None
        self.b2_index: nv.Index | None = None
        self.vecs: Any = None
        self._cache: "OrderedDict[str, tuple[float, nv.Index, Any]]" = OrderedDict()
        self._cache_size = max(2, cache_size)
        self._scratch: dict = {}

    # -- index lifetime ---------------------------------------------------------------------------------------------
    def _build(self, embeddings: Any) -> nv.Index:
        nv.require_device()
        t = _cuda_tensor(embeddings)
        f16 = self.dtype == "f16"
        if self.devices and len(self.devices) > 1:
            want16 = self.dtype == "bf16"
            if t is not None:
                import torch
                want16 = want16 or (self.dtype == "auto" and t.dtype == torch.bfloat16)
            host, code, _ = _to_host_matrix(embeddings, want16, want_f16=f16)
            return MultiDeviceIndex(host, code, self.metric, self.devices)  # type: ignore[return-value]
        if t is not None and t.dim() == 2 and t.device.index == self.device:
            # device hand-off: the encoder's output never visits the host on its way into the index
            import torch
            want = torch.bfloat16 if (self.dtype == "bf16" or (self.dtype == "auto" and t.dtype == torch.bfloat16)) else torch.float32
            want = torch.float16 if f16 else want
            t = t.detach().to(want).contiguous()
            if f16 and t.numel() and not bool(torch.isfinite(t).all()):
                _check_f16_range(np.array([0x7C00], dtype=np.uint16))  # raises the range error
            code = {torch.bfloat16: nv.BF16, torch.float16: nv.F16}.get(want, nv.F32)
            return nv.Index(None, code, self.metric, self.device, on_device_ptr=t.data_ptr(), n=t.shape[0], d=t.shape[1])
        host, code, _ = _to_host_matrix(embeddings, self.dtype == "bf16", want_f16=f16)
        return nv.Index(host, code, self.metric, self.device)

    def _remember(self, index_dir: str, idx: nv.Index, vecs: Any) -> None:
        key = os.path.abspath(index_dir)
        try:
            stamp = os.path.getmtime(f"{index_dir}/index")
        except OSError:
            stamp = 0.0
        old = self._cache.pop(key, None)
        if old is not None and old[1] is not idx:
            old[1].close()
        self._cache[key] = (stamp, idx, vecs)
        while len(self._cache) > self._cache_size:
            _, (_, victim, _) = self._cache.popitem(last=False)
            if victim is not self.b2_index:
                victim.close()

    def index(self, docs: Any, embeddings: Any, index_dir: str, **kwargs: Any) -> None:
        """faiss_vs.py:22-30: build the flat index, persist `vecs` (pickle) and `index` (faiss IndexFlat file)."""
        idx = self._build(embeddings)
        _, _, f32 = _to_host_matrix(embeddings, False)
        faiss_io.write_index_dir(index_dir, embeddings, f32, self.metric, kind=self.factory_string)
        self.b2_index = idx
        self.vecs = embeddings
        self.index_dir = index_dir
        self._remember(index_dir, idx, embeddings)

    def load_index(self, index_dir: str) -> None:
        """faiss_vs.py:32-36. Directories written by FaissVS load unchanged; a device-resident copy is cached per
        directory so operators that alternate between two indexes (sem_sim_join.py:111-127) do not rebuild."""
        key = os.path.abspath(index_dir)
        hit = self._cache.get(key)
        if hit is not None:
            try:
                fresh = os.path.getmtime(f"{index_dir}/index") == hit[0]
            except OSError:
                fresh = False
            if fresh:
                self._cache.move_to_end(key)
                self.index_dir, self.b2_index, self.vecs = index_dir, hit[1], hit[2]
                return
        vecs, x, metric, kind = faiss_io.read_index_dir(index_dir, with_kind=True)
        if metric != self.metric:
            raise ValueError(f"index at {index_dir} was built with metric {metric}, this store uses {self.metric}")
        if kind != self.factory_string:
            raise ValueError(f"index at {index_dir} is a {kind!r} index, this store uses factory_string={self.factory_string!r}")
        idx = self._build(x if (self.sq or self.dtype == "f32") else vecs)
        self.index_dir, self.b2_index, self.vecs = index_dir, idx, vecs
        self._remember(index_dir, idx, vecs)

    # -- queries ----------------------------------------------------------------------------------------------------
    def _entry_for(self, index_dir: str) -> nv.Index:
        """Device index of `index_dir` WITHOUT making it the loaded one (faiss_vs.py:38-41 only reads the `vecs` pickle and
        leaves `self.faiss_index` / `self.index_dir` alone)."""
        key = os.path.abspath(index_dir)
        if self.index_dir is not None and self.b2_index is not None and os.path.abspath(self.index_dir) == key:
            return self.b2_index
        keep = (self.index_dir, self.b2_index, self.vecs)
        if self.index_dir is not None and os.path.abspath(self.index_dir) in self._cache:
            self._cache.move_to_end(os.path.abspath(self.index_dir))  # the loaded index must not be the eviction victim
        try:
            self.load_index(index_dir)  # per-directory cache hit, or build + cache the device copy ...
            return self.b2_index  # type: ignore[return-value]
        finally:
            self.index_dir, self.b2_index, self.vecs = keep  # ... but the loaded index stays what it was

    def get_vectors_from_index(self, index_dir: str, ids: Any) -> np.ndarray:
        """faiss_vs.py:38-41 (`pickle.load(vecs)[ids]`), served by the device row-gather kernel. Like the reference it does
        not change which index is loaded."""
        idx = self._entry_for(index_dir)
        ids_a = np.asarray(list(ids) if not isinstance(ids, np.ndarray) else ids, dtype=np.int64)
        if self.sq:  # SQfp16: the pickle keeps the original embeddings and the reference returns those, not the fp16 rows
            orig = self._originals(index_dir)
            if len(ids_a) and (ids_a.min() < -len(orig) or ids_a.max() >= len(orig)):
                raise IndexError(f"ids contains a position outside [0, {len(orig)})")
            return orig[ids_a]
        out = idx.gather(ids_a)
        if idx.dtype == nv.F16:
            return nv.f16_bits_to_f32(out)
        return BF16Backed.wrap(nv.bf16_bits_to_f32(out)) if idx.dtype == nv.BF16 else out

    def _originals(self, index_dir: str) -> np.ndarray:
        """The `vecs` of `index_dir` (what index() was given) as float32 — faiss casts whatever it is given to float32."""
        key = os.path.abspath(index_dir)
        hit = self._cache.get(key)
        vecs = hit[2] if hit is not None else self.vecs
        return _to_host_matrix(vecs, False)[2]

    def __call__(self, query_vectors: Any, K: int, ids: list[int] | None = None, **kwargs: Any) -> RMOutput:
        """faiss_vs.py:43-77. Returns float32 distances [Q,K] and int64 indices [Q,K] (global ids; -1 = no result).
        The reference's wrap-around of -1 to the last id when K > len(ids) (faiss_vs.py:71-72) is NOT reproduced."""
        if self.b2_index is None or self.index_dir is None:
            raise ValueError("Index not loaded")
        ids_a = None if ids is None else np.asarray(list(ids) if not isinstance(ids, np.ndarray) else ids, dtype=np.int64)
        t = _cuda_tensor(query_vectors)
        if t is not None and ids_a is None and t.dim() == 2 and t.device.index == self.device and not isinstance(self.b2_index, MultiDeviceIndex):
            return self._call_device(t, int(K))
        q, code, _ = _to_host_matrix(query_vectors, False, exact_bf16_ok=self.b2_index.dtype == nv.BF16, scratch=self._scratch,
                                     exact_f16_ok=self.b2_index.dtype == nv.F16)
        if q.shape[1] != self.b2_index.d:
            raise ValueError(f"query dimension {q.shape[1]} does not match the index dimension {self.b2_index.d}")
        try:
            distances, indices = self.b2_index.search(q, int(K), code, ids=ids_a)
        except nv.NativeError as e:
            if e.code in (nv.EINVAL, nv.ERANGE):
                raise ValueError(e.msg) from e
            raise
        return RMOutput(distances=distances, indices=indices)

    def _call_device(self, t: Any, K: int) -> RMOutput:
        """Queries already on the GPU (e.g. straight out of the encoder): search in place, only the [Q,K] result travels."""
        import torch
        assert self.b2_index is not None
        if t.shape[1] != self.b2_index.d:
            raise ValueError(f"query dimension {t.shape[1]} does not match the index dimension {self.b2_index.d}")
        q = t.detach()
        # fp16 queries stream in place against an fp16 store; any other store sees them widened to fp32, as before
        native = (torch.float32, torch.bfloat16, torch.float16) if self.b2_index.dtype == nv.F16 else (torch.float32, torch.bfloat16)
        q = q.contiguous() if q.dtype in native else q.to(torch.float32).contiguous()
        code = {torch.bfloat16: nv.BF16, torch.float16: nv.F16}.get(q.dtype, nv.F32)
        out_s = torch.empty((q.shape[0], K), dtype=torch.float32, device=q.device)
        out_i = torch.empty((q.shape[0], K), dtype=torch.int64, device=q.device)
        try:
            self.b2_index.search_dev(q.data_ptr(), q.shape[0], K, code, out_s.data_ptr(), out_i.data_ptr(),
                                     stream=torch.cuda.current_stream().cuda_stream)
        except nv.NativeError as e:
            if e.code in (nv.EINVAL, nv.ERANGE):
                raise ValueError(e.msg) from e
            raise
        return RMOutput(distances=out_s.cpu().numpy(), indices=out_i.cpu().numpy())

    # -- extensions used by the re-registered operators --------------------------------------------------------------
    def threshold_pairs(self, threshold: float):
        if self.sq:
            # the reference relation x_i . fp16(x_j) > t is asymmetric (fp32 query against the fp16 row); the all-pairs kernel is
            # symmetric. sem_dedup then runs the reference's own relation through __call__ (O(n^2), like the reference).
            raise NotImplementedError("threshold_pairs is not available on an SQfp16 store (asymmetric relation)")
        if self.b2_index is None:
            raise ValueError("Index not loaded")
        return self.b2_index.threshold_pairs(threshold)

    def kmeans(self, ids: Any, ncentroids: int, niter: int = 20, seed: int = 1234, full_lloyd: bool = False):
        if self.b2_index is None:
            raise ValueError("Index not loaded")
        ids_a = np.asarray(ids, dtype=np.int64)
        if self.sq:
            # lotus.utils.cluster trains faiss.Kmeans on get_vectors_from_index, i.e. on the original embeddings: a temporary
            # fp32 index over vecs[ids], not the fp16 rows
            assert self.index_dir is not None
            tmp = nv.Index(np.ascontiguousarray(self._originals(self.index_dir)[ids_a]), nv.F32, self.metric, self.device)
            try:
                return tmp.kmeans(ncentroids, niter=niter, seed=seed, full_lloyd=full_lloyd)
            finally:
                tmp.close()
        return self.b2_index.kmeans(ncentroids, niter=niter, seed=seed, ids=ids_a, full_lloyd=full_lloyd)

    def close(self) -> None:
        for _, idx, _ in self._cache.values():
            idx.close()
        self._cache.clear()
        self.b2_index = None
