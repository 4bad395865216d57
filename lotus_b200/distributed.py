"""Row-sharded flat index across the GPUs of one box (SURVEY §8e): one process per GPU, torch.distributed for the
plumbing. The corpus rows [r*N/G, (r+1)*N/G) live on rank r; queries are replicated; every rank runs the fused
tcgen05 filter + exact finalize on its shard, then ONE all-gather of the per-shard (score, idx) lists over
NCCL/NVLink and a single-kernel k-way merge (b2_merge_topk_dev). No other collective touches the data path.

The reference is single-process (faiss_vs.py); the sharded result is defined as faiss `IndexShards` would define
it: per-shard flat search, then a merge by (score, shard order). It equals the single-index result whenever no
exact fp32 tie straddles rank K across shards (DESIGN.md §Ties)."""
from __future__ import annotations

import os
from typing import Optional

import numpy as np

from . import _native as nv


def shard_bounds(n: int, world: int, rank: int) -> tuple[int, int]:
    """Contiguous row range of `rank`: the first n % world ranks get one extra row."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _torch_code(dtype):
    """Native element-type code of a torch dtype (None for the ones the library does not take)."""
    import torch
    return {torch.float32: nv.F32, torch.bfloat16: nv.BF16, torch.float16: nv.F16}.get(dtype)


class ShardedIndex:
    """Each rank holds `local_rows` (a torch CUDA tensor [n_local, d], fp32, bf16 or fp16) = its slice of the corpus."""

    def __init__(self, local_rows, row_offset: int, metric: int = nv.METRIC_IP, group=None):
        import torch
        import torch.distributed as dist
        self.torch = torch
        self.dist = dist
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        assert local_rows.is_cuda and local_rows.dim() == 2 and local_rows.is_contiguous()
        self.device = local_rows.device.index if local_rows.device.index is not None else torch.cuda.current_device()
        self.dtype = _torch_code(local_rows.dtype)
        if self.dtype is None:
            raise TypeError("corpus must be float32, bfloat16 or float16")
        self.metric = metric
        self.row_offset = int(row_offset)
        n, d = local_rows.shape
        self.index = nv.Index(None, self.dtype, metric, self.device, on_device_ptr=local_rows.data_ptr(), n=n, d=d)
        self.d = d
        self.shard_offsets = np.zeros(self.world, dtype=np.int64)
        if self.world > 1:  # global id of row 0 of every shard (the packed exchange carries local ids)
            t = torch.tensor([self.row_offset], dtype=torch.int64, device=local_rows.device)
            allo = torch.empty(self.world, dtype=torch.int64, device=local_rows.device)
            dist.all_gather_into_tensor(allo, t, group=group)
            self.shard_offsets = allo.cpu().numpy()
        else:
            self.shard_offsets[0] = self.row_offset

    def search(self, q, k: int, ids=None):
        """q: torch CUDA tensor [nq, d] (fp32, bf16 or fp16), replicated on every rank.
        ids: optional GLOBAL row ids (ascending, replicated): each rank keeps those inside its row range — the sharded
        form of FaissVS.__call__(ids=...) (faiss_vs.py:57-72).
        -> (scores [nq,k] float32, idx [nq,k] int64) CUDA tensors holding the GLOBAL top-k on every rank."""
        torch = self.torch
        assert q.is_cuda and q.is_contiguous() and q.shape[1] == self.d
        nq = q.shape[0]
        q_dtype = _torch_code(q.dtype)
        if q_dtype is None:
            raise TypeError("queries must be float32, bfloat16 or float16")
        stream = torch.cuda.current_stream().cuda_stream
        if ids is None and self.world > 1:
            return self._search_packed(q, k)
        loc_s = torch.empty((nq, k), dtype=torch.float32, device=q.device)
        loc_i = torch.empty((nq, k), dtype=torch.int64, device=q.device)
        if ids is not None:
            ids_t = torch.as_tensor(np.asarray(ids, dtype=np.int64), device=q.device)
            mine = ids_t[(ids_t >= self.row_offset) & (ids_t < self.row_offset + self.index.n)] - self.row_offset
            mine = mine.contiguous()
            torch.cuda.current_stream().synchronize()
            self.index.search_dev(q.data_ptr(), nq, k, q_dtype, loc_s.data_ptr(), loc_i.data_ptr(),
                                  ids_ptr=mine.data_ptr() if mine.numel() else None, n_ids=int(mine.numel()), stream=stream)
            if mine.numel() == 0:
                loc_s.fill_(-3.4028234663852886e38 if self.metric == nv.METRIC_IP else 3.4028234663852886e38)
                loc_i.fill_(-1)
            loc_i = torch.where(loc_i >= 0, loc_i + self.row_offset, loc_i)
        else:
            self.index.search_dev(q.data_ptr(), nq, k, q_dtype, loc_s.data_ptr(), loc_i.data_ptr(),
                                  id_offset=self.row_offset, stream=stream)
        if self.world == 1:
            return loc_s, loc_i
        all_s = torch.empty((self.world, nq, k), dtype=torch.float32, device=q.device)
        all_i = torch.empty((self.world, nq, k), dtype=torch.int64, device=q.device)
        self.dist.all_gather_into_tensor(all_s, loc_s, group=self.group)
        self.dist.all_gather_into_tensor(all_i, loc_i, group=self.group)
        out_s = torch.empty_like(loc_s)
        out_i = torch.empty_like(loc_i)
        nv.merge_topk_dev(all_s.data_ptr(), all_i.data_ptr(), self.world, nq, k, self.metric, self.device,
                          out_s.data_ptr(), out_i.data_ptr(), stream=stream)
        return out_s, out_i

    def _search_packed(self, q, k: int):
        """The whole-index step: local search -> ONE all-gather of 8-byte (score, local id) entries -> single-kernel k-way merge."""
        torch = self.torch
        nq = q.shape[0]
        q_dtype = _torch_code(q.dtype)
        stream = torch.cuda.current_stream().cuda_stream
        timing = os.environ.get("B2_SHARD_TIMING") == "1"
        if timing:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            ev[0].record()
        loc = torch.empty((nq, k), dtype=torch.int64, device=q.device)  # uint64 words (torch has no uint64 collectives)
        if os.environ.get("B2_SHARD_STAGED", "1") != "0":
            # two stages: filter, tell the other ranks how good this shard's best ceil(k/G) candidates are (one all-reduce MIN of
            # nq floats), then re-score only what can still reach the merged top k
            lower = torch.empty(nq, dtype=torch.float32, device=q.device)
            self.index.search_stage1_dev(q.data_ptr(), nq, k, q_dtype, -(-k // self.world), lower.data_ptr(), stream=stream)
            self.dist.all_reduce(lower, op=self.dist.ReduceOp.MIN, group=self.group)
            self.index.search_stage2_packed_dev(lower.data_ptr(), loc.data_ptr(), stream=stream)
        else:
            self.index.search_packed_dev(q.data_ptr(), nq, k, q_dtype, loc.data_ptr(), stream=stream)
        if timing:
            ev[1].record()
        allp = torch.empty((self.world, nq, k), dtype=torch.int64, device=q.device)
        self.dist.all_gather_into_tensor(allp, loc, group=self.group)
        if timing:
            ev[2].record()
        out_s = torch.empty((nq, k), dtype=torch.float32, device=q.device)
        out_i = torch.empty((nq, k), dtype=torch.int64, device=q.device)
        nv.merge_topk_packed_dev(allp.data_ptr(), self.shard_offsets, self.world, nq, k, self.metric, self.device,
                                 out_s.data_ptr(), out_i.data_ptr(), stream=stream)
        if timing:
            ev[3].record()
            torch.cuda.synchronize()
            self.last_phase_ms = {"search (filter + finalize + pack)": ev[0].elapsed_time(ev[1]), "filter kernel": self.index.last_filter_ms(),
                                  "all_gather (+ wait for the slowest rank)": ev[1].elapsed_time(ev[2]), "merge": ev[2].elapsed_time(ev[3])}
        return out_s, out_i

    def search_host(self, q_host, k: int, out_scores_host=None, out_idx_host=None):
        """End-to-end form: `q_host` is the (pinned) host query batch [nq, d], present in every rank's process. Each rank copies
        only ITS 1/world slice over PCIe and the ranks all-gather the slices over NVLink; rank 0 (or every rank when the output
        buffers are given there) copies the merged result back. Returns the device tensors (scores, idx)."""
        torch = self.torch
        nq = q_host.shape[0]
        dev = torch.device("cuda", self.device)
        if self.world == 1:
            q = q_host.to(dev, non_blocking=True)
        else:
            per = -(-nq // self.world)
            lo, hi = min(self.rank * per, nq), min((self.rank + 1) * per, nq)
            part = torch.zeros((per, q_host.shape[1]), dtype=q_host.dtype, device=dev)
            if hi > lo:
                part[:hi - lo].copy_(q_host[lo:hi], non_blocking=True)
            full = torch.empty((self.world * per, q_host.shape[1]), dtype=q_host.dtype, device=dev)
            self.dist.all_gather_into_tensor(full, part, group=self.group)
            q = full[:nq]
        s, i = self.search(q, k)
        if out_scores_host is not None:
            out_scores_host.copy_(s, non_blocking=True)
            out_idx_host.copy_(i, non_blocking=True)
        return s, i

    def last_filter_ms(self) -> float:
        return self.index.last_filter_ms()

    def close(self) -> None:
        self.index.close()


def merge_host_lists(scores: np.ndarray, idx: np.ndarray, metric: int):
    """Host restatement of the k-way merge rule (used by the gloo CPU tests of the sharding logic only):
    scores/idx [g, nq, k], lists sorted best first -> [nq, k]. Equal scores: L2 keeps list order from the lowest
    shard up; IP from the highest shard down (faiss's heap order, see DESIGN.md §Ties)."""
    g, nq, k = scores.shape
    out_s = np.empty((nq, k), dtype=np.float32)
    out_i = np.empty((nq, k), dtype=np.int64)
    pad = np.finfo(np.float32).max if metric == nv.METRIC_L2 else -np.finfo(np.float32).max
    for q in range(nq):
        ent = []
        for gi in range(g):
            for p in range(k):
                if idx[gi, q, p] >= 0:
                    s = float(scores[gi, q, p])
                    tie = gi * k + p if metric == nv.METRIC_L2 else (g - 1 - gi) * k + p
                    ent.append(((s if metric == nv.METRIC_L2 else -s), tie, gi, p))
        ent.sort(key=lambda e: (e[0], e[1]))
        for o in range(k):
            if o < len(ent):
                _, _, gi, p = ent[o]
                out_s[q, o] = scores[gi, q, p]
                out_i[q, o] = idx[gi, q, p]
            else:
                out_s[q, o] = pad
                out_i[q, o] = -1
    return out_s, out_i


# ---- multi-GPU dedup and k-means (SURVEY.md §8e) ----------------------------------------------------------------------
def sharded_threshold_pairs(index: "nv.Index", threshold: float, group=None):
    """All pairs i<j with score > threshold when EVERY rank holds the full corpus in `index` (it fits: 7.7 GB for
    10M x 384 bf16): the upper-triangular tile grid is dealt to the ranks in groups of 148 query tiles (`part`/`nparts` of
    b2_threshold_pairs), each rank filters + verifies its tiles, then one all-gather of the sparse pair lists.
    Returns the same (pi, pj) — sorted by (i, j) — on every rank."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if world > 1 else 0
    pi, pj = index.threshold_pairs(threshold, part=rank, nparts=world)
    if world == 1:
        return pi, pj
    dev = torch.device("cuda", index.device) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    cnt = torch.tensor([len(pi)], dtype=torch.int64, device=dev)
    cnts = [torch.zeros_like(cnt) for _ in range(world)]
    dist.all_gather(cnts, cnt, group=group)
    cap = int(max(int(c.item()) for c in cnts))
    buf = torch.full((2, max(cap, 1)), -1, dtype=torch.int64, device=dev)
    buf[0, :len(pi)] = torch.from_numpy(pi).to(dev)
    buf[1, :len(pj)] = torch.from_numpy(pj).to(dev)
    bufs = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(bufs, buf, group=group)
    ai = np.concatenate([b[0, :int(c.item())].cpu().numpy() for b, c in zip(bufs, cnts)])
    aj = np.concatenate([b[1, :int(c.item())].cpu().numpy() for b, c in zip(bufs, cnts)])
    order = np.lexsort((aj, ai))
    return ai[order], aj[order]


def sharded_kmeans(index: "nv.Index", n_total: int, row_offset: int, k: int, niter: int = 20, seed: int = 1234, group=None,
                   want_obj: bool = True):
    """Full-Lloyd k-means over points row-sharded across ranks (`index` holds this rank's rows [row_offset, row_offset+n_local)).
    faiss's control flow (lotus/utils.py:61-65 -> faiss/Clustering.cpp): initial centroids = the first k points of
    rand_perm(n_total, seed+1) (fetched from whichever rank owns them), then per iteration, all on the device:
    exact assignment of the local points (b2_kmeans_assign_dev), per-shard point-order fp32 sums + counts (+ the fp64
    objective) in one pass (b2_kmeans_accumulate_dev), ONE NCCL all-reduce(sum) of the packed [k,d] sums | [k] counts,
    division; split_clusters is replayed identically on every rank in the (rare) iterations that leave a cluster empty.
    The cross-rank fp32 reduction makes centroids agree with the single-process restatement to rounding, not bit-for-bit
    (DESIGN.md §6). Returns (local assignment [n_local] int64, centroids [k,d] float32, objective per iteration) as numpy."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    dev = torch.device("cuda", index.device)
    n_local, d = index.n, index.d
    stream = torch.cuda.current_stream(dev).cuda_stream
    # initial centroids: rows perm[:k] of the global matrix (only the first k steps of the Fisher-Yates shuffle are needed)
    raw = np.random.RandomState((seed + 1) & 0xFFFFFFFF)._bit_generator.random_raw(max(min(k, n_total), 1))  # std::mt19937 stream
    moved: dict[int, int] = {}
    want = np.empty(k, dtype=np.int64)
    for i in range(k):
        if i + 1 < n_total:
            i2 = i + int(raw[i]) % (n_total - i)
            a, b = moved.get(i, i), moved.get(i2, i2)
            moved[i], moved[i2] = b, a
        want[i] = moved.get(i, i)
    mine = (want >= row_offset) & (want < row_offset + n_local)
    cent_h = np.zeros((k, d), dtype=np.float32)
    if mine.any():
        rows = index.gather(want[mine] - row_offset)
        cent_h[mine] = nv.bits_to_f32(rows, index.dtype)
    cent = torch.from_numpy(cent_h).to(dev)
    if world > 1:
        dist.all_reduce(cent, group=group)  # each row is non-zero on exactly one rank
    packed = torch.empty(k * d + k, dtype=torch.float32, device=dev)
    sums, counts = packed[:k * d].view(k, d), packed[k * d:]
    assign = torch.empty(max(n_local, 1), dtype=torch.int64, device=dev)
    obj = torch.zeros(max(niter, 1), dtype=torch.float64, device=dev)
    for it in range(niter):
        index.kmeans_assign_dev(cent.data_ptr(), k, assign.data_ptr(), stream=stream)
        index.kmeans_accumulate_dev(assign.data_ptr(), k, sums.data_ptr(), counts.data_ptr(),
                                    centroids_ptr=cent.data_ptr() if want_obj else 0,
                                    obj_ptr=obj[it:].data_ptr() if want_obj else 0, stream=stream)
        if world > 1:
            dist.all_reduce(packed, group=group)
        nz = counts > 0
        inv = torch.reciprocal(torch.where(nz, counts, torch.ones_like(counts)))  # fp32 1/count, then one fp32 multiply: faiss's order
        cent = torch.where(nz[:, None], sums * inv[:, None], torch.zeros_like(sums)).contiguous()
        if not bool(nz.all()):
            c_h, _ = split_clusters_host(cent.cpu().numpy(), counts.cpu().numpy(), n_total)
            cent = torch.from_numpy(c_h).to(dev)
    if world > 1 and want_obj and niter > 0:
        dist.all_reduce(obj, group=group)
    index.kmeans_assign_dev(cent.data_ptr(), k, assign.data_ptr(), stream=stream)  # same stream as the torch ops: ordered
    return assign[:n_local].cpu().numpy(), cent.cpu().numpy(), obj[:niter].to(torch.float32).cpu().numpy()


def split_clusters_host(centroids: np.ndarray, hassign: np.ndarray, n: int):
    """faiss/Clustering.cpp split_clusters (EPS = 1/1024, RandomGenerator rng(1234)) on host arrays; every rank replays
    the same stream so the replicated centroids stay identical."""
    c = np.ascontiguousarray(centroids, dtype=np.float32).copy()
    h = np.ascontiguousarray(hassign, dtype=np.float32).copy()
    k, d = c.shape
    raw = iter(np.random.RandomState(1234)._bit_generator.random_raw(1 << 16).tolist())
    eps = 1 / 1024.0
    even = (np.arange(d) % 2 == 0)
    for ci in range(k):
        if h[ci] == 0:
            cj = 0
            while True:
                p = np.float32((np.float64(h[cj]) - 1.0) / np.float64(np.float32(n - k)))
                r = np.float32(next(raw)) / np.float32(4294967295)
                if r < p:
                    break
                cj = (cj + 1) % k
            base = c[cj].astype(np.float64)
            c[ci] = np.where(even, base * (1 + eps), base * (1 - eps)).astype(np.float32)
            c[cj] = np.where(even, base * (1 - eps), base * (1 + eps)).astype(np.float32)
            h[ci] = h[cj] / 2
            h[cj] -= h[ci]
    return c, h
