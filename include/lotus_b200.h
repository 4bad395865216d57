/*
 * lotus_b200.h — C-ABI of libb2lotus.so, the B200 (sm_100a) vector-store backend for LOTUS.
 *
 * This is the drop-in boundary for ONE hot path of lotus-data/lotus: the faiss-backed
 * `lotus.vector_store.FaissVS` and the faiss.Kmeans call in `lotus.utils.cluster`.
 * Every entry point below replaces one faiss call site of the reference (citations are
 * relative to the reference tree, lotus-data/lotus @ 136ae4f4):
 *
 *   b2_index_create        <- faiss.index_factory + Index.add      lotus/vector_store/faiss_vs.py:23-24, :63-64
 *   b2_index_search        <- Index.search (whole index)           lotus/vector_store/faiss_vs.py:75
 *                             tmp_index.search + id remap (ids=)   lotus/vector_store/faiss_vs.py:57-72
 *   b2_index_gather        <- pickle.load(vecs)[ids]               lotus/vector_store/faiss_vs.py:38-41
 *   b2_threshold_pairs     <- sem_sim_join(K=N) + `_scores > thr`  lotus/sem_ops/sem_dedup.py:45-46
 *   b2_connected_components<- DFS over the pair set                lotus/sem_ops/sem_dedup.py:58-84
 *   b2_kmeans              <- faiss.Kmeans(d,k,niter).train +
 *                             kmeans.index.search(x, 1)            lotus/utils.py:61-65
 *   b2_merge_topk_dev      <- (no reference call site: the reference is single process; this is the
 *                             k-way merge after the NCCL all-gather of per-shard candidates)
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / CUDA types in any signature (a stream is passed as void*).
 *   - every function returns 0 on success, a negative B2_E* code on failure; the message for the calling
 *     thread's last failure is b2_last_error().
 *   - "host" entry points take HOST buffers and do their own H2D/D2H copies (these are what a plugin calls);
 *     "_dev" entry points take DEVICE buffers that live on the index's device, enqueue on `stream`
 *     (a cudaStream_t cast to void*, NULL = the legacy default stream) and return after the results are
 *     complete in the output buffers (they synchronise `stream` before returning).
 *   - the caller owns every in/out buffer; the library owns the b2_index handle and its device memory.
 *   - one in-flight call per handle (the reference's FaissVS is not re-entrant either).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point returns B2_ENODEV.
 *
 * Result semantics (identical to faiss IndexFlatIP / IndexFlatL2 as restated in oracle/faiss_flat.c):
 *   - metric IP: larger is better, rows sorted best first; metric L2: squared distance, ascending.
 *   - fewer than k results: index -1 and score -FLT_MAX (IP) / +FLT_MAX (L2).
 *   - scores are the canonical fp32 score: the dot product (or sum of squared differences) accumulated
 *     in fp64 in a fixed order and rounded once to fp32 (see oracle/faiss_flat.c `orc_dot_canonical`).
 *   - exact ties follow faiss's heap (utils/Heap.h): L2 -> (dist asc, id asc); IP -> (score desc, id desc),
 *     with the retention window at rank k described in DESIGN.md §Ties.
 */
#ifndef LOTUS_B200_H
#define LOTUS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_ABI_VERSION 1

#if defined(__GNUC__)
#define B2_API __attribute__((visibility("default")))
#else
#define B2_API
#endif

/* element types of embedding matrices (B2_F16: IEEE binary16, the storage of faiss's "SQfp16"). Every entry point that takes
 * a store dtype or a q_dtype accepts all three, in any combination. */
enum { B2_F32 = 0, B2_BF16 = 1, B2_F16 = 2 };
/* metrics; numeric values match faiss.METRIC_INNER_PRODUCT / faiss.METRIC_L2 */
enum { B2_METRIC_IP = 0, B2_METRIC_L2 = 1 };

/* error codes */
enum {
    B2_OK = 0,
    B2_EINVAL = -1,   /* bad argument */
    B2_ENODEV = -2,   /* no CUDA device / wrong architecture */
    B2_ECUDA = -3,    /* CUDA runtime or driver error */
    B2_ENOMEM = -4,   /* allocation failed */
    B2_ERANGE = -5    /* k or an id out of the supported range */
};

typedef struct b2_index b2_index;

/* ---- library ---------------------------------------------------------------------------------------- */
B2_API int b2_abi_version(void);
B2_API const char* b2_last_error(void);
/* number of visible CUDA devices that are sm_100 (B200); 0 when there is none */
B2_API int b2_device_count(void);
/* largest k supported by b2_index_search */
B2_API int b2_max_k(void);

/* ---- index lifetime (faiss_vs.py:22-36) -------------------------------------------------------------- */
/* Build a flat index over x[n,d] (row-major, `dtype` elements). x is a HOST pointer unless x_on_device != 0.
 * The matrix is copied; the caller may free x afterwards. */
B2_API int b2_index_create(const void* x, int64_t n, int32_t d, int32_t dtype, int32_t metric, int32_t device,
                    int32_t x_on_device, b2_index** out);
B2_API void b2_index_free(b2_index* idx);
B2_API int64_t b2_index_ntotal(const b2_index* idx);
B2_API int32_t b2_index_dim(const b2_index* idx);
B2_API int32_t b2_index_dtype(const b2_index* idx);
B2_API int32_t b2_index_metric(const b2_index* idx);
B2_API int32_t b2_index_device(const b2_index* idx);
/* device pointer of the stored matrix [n,d] in `dtype` (for zero-copy hand-off to torch) */
B2_API const void* b2_index_data_dev(const b2_index* idx);

/* ---- search (faiss_vs.py:43-77) ---------------------------------------------------------------------- */
/* q[nq,d] in q_dtype. ids == NULL: search the whole index. ids != NULL (n_ids entries, positions into the
 * index, any order): search only those rows and report the ORIGINAL ids (the reference builds a temporary
 * index over vecs[ids] and remaps; ties follow the order of `ids`).
 * out_scores[nq,k] float32, out_idx[nq,k] int64. HOST buffers. */
B2_API int b2_index_search(b2_index* idx, const void* q, int64_t nq, int32_t q_dtype, int32_t k, const int64_t* ids,
                    int64_t n_ids, float* out_scores, int64_t* out_idx);

/* DEVICE buffers; ids_dev may be NULL. id_offset is added to every reported id when ids_dev == NULL
 * (row-sharded multi-GPU: global id = local id + shard offset). */
B2_API int b2_index_search_dev(b2_index* idx, const void* q_dev, int64_t nq, int32_t q_dtype, int32_t k,
                        const int64_t* ids_dev, int64_t n_ids, int64_t id_offset, float* out_scores_dev,
                        int64_t* out_idx_dev, void* stream);

/* k-way merge of g per-shard result lists: scores[g,nq,k], idx[g,nq,k] (each list sorted best first, shard
 * s holding ids below those of shard s+1) -> out[nq,k]. DEVICE buffers on `device`. */
B2_API int b2_merge_topk_dev(const float* scores_dev, const int64_t* idx_dev, int32_t g, int64_t nq, int32_t k,
                      int32_t metric, int32_t device, float* out_scores_dev, int64_t* out_idx_dev, void* stream);

/* The same two steps with ONE 8-byte word per entry — (float32 score bits << 32) | local row id, 0xffffffff = no result — so
 * the row-sharded exchange is a single all-gather of nq*k*8 bytes per rank (25.6 MB at 100k x 32) instead of scores + int64 ids
 * (38 MB in two collectives). b2_index_search_packed_dev searches the whole index and reports LOCAL ids;
 * b2_merge_topk_packed_dev takes packed[g,nq,k] plus shard_offsets[g] (HOST array: global id of row 0 of shard s) and writes
 * float32 scores and int64 GLOBAL ids. */
B2_API int b2_index_search_packed_dev(b2_index* idx, const void* q_dev, int64_t nq, int32_t q_dtype, int32_t k,
                               uint64_t* out_packed_dev, void* stream);
B2_API int b2_merge_topk_packed_dev(const uint64_t* packed_dev, const int64_t* shard_offsets, int32_t g, int64_t nq, int32_t k,
                             int32_t metric, int32_t device, float* out_scores_dev, int64_t* out_idx_dev, void* stream);

/* Row-sharded search in two stages, so that the ranks can tell each other how good the merged top k will be BEFORE the exact
 * re-scoring. Stage 1 filters this shard (tcgen05 kernel) and writes lower_dev[nq]: for every query a lower bound on the exact
 * score of its j best local candidates (-inf when unknown); it only enqueues work on `stream`. The caller all-reduces (MIN)
 * lower_dev over the ranks with j = ceil(k / ranks) — k rows of the whole index are then known to reach that score — and hands
 * the result to stage 2, which re-scores only the local candidates that can still reach it (about k / ranks instead of k + 2),
 * certifies against it, and writes the packed [nq,k] list like b2_index_search_packed_dev. q_dev must stay valid until
 * stage 2 returns. One staged search in flight per handle. */
B2_API int b2_index_search_stage1_dev(b2_index* idx, const void* q_dev, int64_t nq, int32_t q_dtype, int32_t k, int32_t j,
                               float* lower_dev, void* stream);
B2_API int b2_index_search_stage2_packed_dev(b2_index* idx, const float* hint_dev, uint64_t* out_packed_dev, void* stream);

/* ---- row gather (faiss_vs.py:38-41) ------------------------------------------------------------------ */
/* out[m,d] in the index's dtype = x[ids]; HOST out unless out_on_device != 0 (then ids is a device pointer too) */
B2_API int b2_index_gather(b2_index* idx, const int64_t* ids, int64_t m, void* out, int32_t out_on_device);

/* ---- dedup (sem_dedup.py:45-84) ---------------------------------------------------------------------- */
/* All unordered pairs i<j with canonical score(i,j) > threshold (IP; strict, as sem_dedup.py:46).
 * out_i/out_j: HOST arrays of capacity cap; *n_pairs receives the number found (may exceed cap: then only the
 * first cap pairs in (i,j) order are stored and the call returns B2_ERANGE).
 * part/nparts: process only the row-tile slice `part` of `nparts` (multi-GPU sharding of the pair space);
 * pass 0,1 for everything. Pairs are returned sorted by (i,j). */
B2_API int b2_threshold_pairs(b2_index* idx, float threshold, int32_t part, int32_t nparts, int64_t* out_i,
                       int64_t* out_j, int64_t cap, int64_t* n_pairs);
/* labels[n] = smallest row id of the connected component of each row under the pair list (HOST buffers). */
B2_API int b2_connected_components(int64_t n, const int64_t* pi, const int64_t* pj, int64_t n_pairs, int32_t device,
                            int64_t* labels);

/* ---- k-means (lotus/utils.py:61-65) ------------------------------------------------------------------ */
/* faiss.Kmeans(d, k, niter=niter, seed=1234, max_points_per_centroid=256).train(x[ids]) followed by
 * index.search(x[ids], 1). ids may be NULL (all rows). out_assign[m] int64, out_centroids[k,d] float32
 * (nullable), out_obj[niter] float32 (nullable, the objective of every iteration). HOST buffers.
 * full_lloyd != 0 trains on every point instead of faiss's 256*k subsample. */
B2_API int b2_kmeans(b2_index* idx, const int64_t* ids, int64_t m, int32_t k, int32_t niter, int64_t seed,
              int32_t full_lloyd, int64_t* out_assign, float* out_centroids, float* out_obj);
/* one assignment pass against given centroids[k,d] (float32, HOST): out_assign[m] int64, out_dist[m] float32
 * (nullable). This is `kmeans.index.search(x, 1)` with explicit centroids. */
B2_API int b2_kmeans_assign(b2_index* idx, const int64_t* ids, int64_t m, const float* centroids, int32_t k,
                     int64_t* out_assign, float* out_dist);

/* DEVICE-buffer forms for the row-sharded multi-GPU Lloyd loop (lotus_b200/distributed.py sharded_kmeans): nothing visits
 * the host between the assignment, the per-shard sums and the NCCL all-reduce of [k,d] sums + [k] counts.
 * b2_kmeans_assign_dev: assign_dev[m] int64 (and dist_dev[m] float32 when non-NULL: the canonical distance to the winner)
 * for the rows ids_dev[0..m) (NULL = all rows) against centroids_dev[k,d] float32.
 * b2_kmeans_accumulate_dev: sums_dev[k,d] float32 = per-centroid sums of the member rows in point order (NOT divided),
 * counts_dev[k] float32; when obj_dev is non-NULL, *obj_dev += sum of squared distances of the rows to
 * centroids_dev[assign] (float64; centroids_dev = the centroids the assignment was made against).
 * All pointers live on the index's device; both calls enqueue on `stream` and synchronise it before returning. */
B2_API int b2_kmeans_assign_dev(b2_index* idx, const int64_t* ids_dev, int64_t m, const float* centroids_dev, int32_t k,
                         int64_t* assign_dev, float* dist_dev, void* stream);
B2_API int b2_kmeans_accumulate_dev(b2_index* idx, const int64_t* ids_dev, int64_t m, const int64_t* assign_dev, int32_t k,
                             const float* centroids_dev, float* sums_dev, float* counts_dev, double* obj_dev, void* stream);

/* per-shard centroid update for multi-GPU Lloyd: for the rows ids[0..m) (or all) and their assignment assign[m],
 * out_sums[k,d] float32 = sum of the member rows of each centroid (point order, fp32, NOT divided), out_counts[k] float32.
 * The caller all-reduces sums and counts over the ranks and divides. HOST buffers. (faiss/Clustering.cpp compute_centroids
 * before its normalisation loop; lotus/utils.py:61-62 calls it through faiss.Kmeans.train.) */
B2_API int b2_kmeans_accumulate(b2_index* idx, const int64_t* ids, int64_t m, const int64_t* assign, int32_t k, float* out_sums,
                         float* out_counts);

/* ---- host-side marshalling (no device work) ------------------------------------------------------------ */
/* out[i] = bfloat16 bit pattern of x[i] (round to nearest even, NaN stays a quiet NaN); *all_exact (nullable) = 1 when
 * every x[i] was already bfloat16-representable, i.e. the 2-byte form loses nothing. The plugin uses it to ship query
 * vectors that came out of a bf16 index (faiss_vs.py:38-41 -> sem_sim_join.py:130-134) in their exact 2-byte form. */
B2_API int b2_host_f32_to_bf16(const float* x, int64_t count, uint16_t* out, int32_t* all_exact);
/* the exact inverse: out[i] = float32 value of the bfloat16 bit pattern x[i] (row gathers of a bf16 index, faiss_vs.py:38-41) */
B2_API int b2_host_bf16_to_f32(const uint16_t* x, int64_t count, float* out);

/* The filter kernel's work schedule for a shape (no device work; used by the CPU tests): kp = candidate-list capacity (0 = the
 * shape goes to the dense path), n_splits = corpus splits, units_whole = leading query units that sweep the whole corpus as one
 * item each (two-phase schedule), two_cta = CTA-pair mode. */
B2_API int b2_debug_filter_plan(int64_t nq, int64_t n, int32_t k, int32_t num_sms, int32_t* kp, int32_t* n_splits,
                         int32_t* units_whole, int32_t* two_cta);

/* ---- instrumentation ---------------------------------------------------------------------------------- */
/* counters since the last b2_stats_reset(): [0] kernels launched by this library, [1] queries answered,
 * [2] queries that took the exact dense fallback, [3] tcgen05 filter launches, [4] rows rescored exactly,
 * [5] queries of fp32 indexes that the bf16 first-level filter could not certify and the tf32 level answered.
 * Returns how many counters were written (<= cap). */
B2_API int b2_stats(int64_t* out, int32_t cap);
B2_API void b2_stats_reset(void);
/* device time (ms) of the dominant kernel (the tcgen05 filter) in the last search on this handle, measured
 * with CUDA events on the stream it was launched on; <0 when unavailable. */
B2_API float b2_last_filter_ms(const b2_index* idx);

#ifdef __cplusplus
}
#endif
#endif /* LOTUS_B200_H */
