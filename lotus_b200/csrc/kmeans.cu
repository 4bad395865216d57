// kmeans.cu — sem_cluster_by's core: faiss.Kmeans(d, k, niter).train(x) followed by kmeans.index.search(x, 1)
// (lotus/utils.py:61-65). The algorithm is faiss/Clustering.cpp's, as oracle/faiss_flat.c `orc_kmeans` restates it:
//   host control flow : subsample to 256*k points with rand_perm(seed) (std::mt19937), initial centroids = first k of
//                       rand_perm(seed+1), niter Lloyd iterations, split_clusters with RandomGenerator(1234)
//   assignment        : argmin_c ||x - c||^2, ties -> lowest centroid id, decided on the canonical (fp64-accumulated) distance
//   centroid update   : faiss sums the member points in POINT ORDER in fp32 and scales by 1/count -> bit-identical centroids
//
// Device pipeline of one Lloyd iteration (everything stays on the device; the only host round trip is one 4-byte counter):
//   1. centroid view  : bf16 (or tf32) filter copy of the fp32 centroids + canonical squared norms + max norm (device scalar)
//   2. filter         : knn_filter_kernel<16, L2, ., ., TOP1> — tcgen05 scores of every point against every centroid, the
//                       epilogue keeps each point's best two centroids and the third-best score in registers
//   3. km_assign_finalize_kernel (thread per point): winner c1 by filter score, runner-up bound f2 (second best, third-best
//                       bounds of every list). |filter - exact| <= eps for every centroid, so f1 - f2 > 2 eps (+ fp32 rounding
//                       slack) PROVES c1 is the exact argmin with no tie: assigned without touching the point again.
//                       Points that cannot be proven are appended to a device list ...
//   4. second level   : ... gathered and answered by the general exact pipeline (search_core: KP=16 lists, canonical re-score,
//                       certificate, dense fallback) and scattered back. Typically < 2 % of the points, ~0 after a few iterations.
//   5. update         : stable counting sort of the points by centroid (member lists in point order), then one warp per
//                       (centroid, 16-byte column chunk) adds its members sequentially with 8 row loads in flight; the same pass
//                       accumulates the objective (sum of exact distances to the OLD centroids, fp64) when it is asked for.
//   6. km_split_kernel: faiss's split_clusters on the device (one block; a device MT19937 replays RandomGenerator(1234)).
#include <algorithm>
#include <chrono>
#include <random>
#include <unordered_map>
#include <vector>

#include "canonical.cuh"
#include "index.cuh"

namespace b2 {

struct KmWork {
    DevBuf cent[2], cent_filt, cent_norm2, scalar, pts, pts_norm2, train, train_norm2, assign, members, offsets, totals, blk, hassign, ids,
        obj, flag_ids, flag_count, hard_ids, order, dbg, sub, sub_dis, sub_assign, fin_assign, fin_dis, perm;
    HostBuf h_count;
    void release() {
        DevBuf* all[] = {&cent[0], &cent[1], &cent_filt, &cent_norm2, &scalar, &pts, &pts_norm2, &train, &train_norm2, &assign, &members,
                         &offsets, &totals, &blk, &hassign, &ids, &obj, &flag_ids, &flag_count, &hard_ids, &order, &dbg, &sub, &sub_dis, &sub_assign, &fin_assign,
                         &fin_dis, &perm};
        for (DevBuf* b : all) b->release();
        h_count.release();
    }
};

void km_work_free(KmWork* w) {
    if (!w) return;
    w->release();
    delete w;
}

namespace {

// First `take` entries of faiss/utils/random.cpp rand_perm(n, seed): Fisher-Yates with rng.rand_int(n - i) = mt() % (n - i).
// Entry i is final after step i, so only `take` steps are replayed, over a sparse view of the (otherwise identity) array.
void rand_perm_prefix(std::vector<int64_t>& out, int64_t n, int64_t take, int64_t seed) {
    out.resize(take);
    std::mt19937 mt((unsigned int)seed);
    std::unordered_map<int64_t, int64_t> moved;
    moved.reserve((size_t)take * 2);
    auto at = [&](int64_t i) {
        auto it = moved.find(i);
        return it == moved.end() ? i : it->second;
    };
    for (int64_t i = 0; i < take; ++i) {
        if (i + 1 < n) {
            const int64_t i2 = i + (int64_t)(mt() % (uint32_t)(n - i));
            const int64_t a = at(i), b = at(i2);
            moved[i] = b;
            moved[i2] = a;
        }
        out[i] = at(i);
    }
}

__global__ void rows_to_f32_kernel(const void* x, int dtype, int d, const int64_t* ids, int64_t m, float* out) {
    const int64_t total = m * d;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = t / d;
        const int c = (int)(t - r * d);
        const int64_t src = ids ? ids[r] : r;
        out[t] = elem_f32(x, dtype, (size_t)(src * d + c));
    }
}

// ---- step 3: decide the assignment from the filter's top-2 lists ---------------------------------------------------------
// cand_* hold, per point and per list (2 epilogue sets x n_splits), the best two (score, centroid) pairs in slots 0-1 and the
// third-best score in cand_thr (-inf when the list saw fewer than three centroids). score = 2 x.c - ||c||^2 (larger = nearer).
__global__ void km_assign_finalize_kernel(const float* cand_score, const int32_t* cand_id, const float* cand_thr, int64_t m, int n_lists,
                                          int list_len, const float* pnorm2, const float* max_norm_dev, float rel_eps, float abs_eps, int64_t* assign,
                                          int32_t* flag_local, int32_t* flag_count, int64_t base) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= m) return;
    float f1 = -INFINITY, f2 = -INFINITY;
    int32_t c1 = -1;
    for (int l = 0; l < n_lists; ++l) {
        const size_t off = ((size_t)i * n_lists + l) * list_len;
        const float2 s = *reinterpret_cast<const float2*>(cand_score + off);
        const int2 id = *reinterpret_cast<const int2*>(cand_id + off);
        if (id.x >= 0) {
            if (s.x > f1) {
                f2 = f1;
                f1 = s.x;
                c1 = id.x;
            } else {
                f2 = fmaxf(f2, s.x);  // an equal score is a potential tie: it closes the gap to zero
            }
        }
        if (id.y >= 0) f2 = fmaxf(f2, s.y);
        f2 = fmaxf(f2, cand_thr[(size_t)i * n_lists + l]);
    }
    const double mx = (double)__ldg(max_norm_dev);
    const double qn2 = (double)pnorm2[base + i];
    const double qn = sqrt(qn2);
    // |filter score - exact score| for any centroid (same bound as finalize_kernel's L2 certificate)
    const double eps_s = 2.0 * filter_ip_err((double)rel_eps, (double)abs_eps, qn, mx) + 2.4e-7 * (mx * mx + 2.0 * qn * mx) + 1e-30;
    // the reported distances are fp32 roundings of ||x||^2 - score: two exact scores further apart than this cannot round equal
    const double slack = 2.4e-7 * (qn2 + fmax(fabs((double)f1), fabs((double)f2)));
    const bool certain = c1 >= 0 && ((double)f1 - (double)f2) > 2.0 * eps_s + slack;  // false for NaN scores as well
    assign[base + i] = c1;
    if (!certain) flag_local[atomicAdd(flag_count, 1)] = (int32_t)i;
}

// ---- step 4a: points the gap test left open, decided among their KNOWN contenders -------------------------------------------
// Warp per flagged point. Every centroid whose exact score could reach the winner's is either one of the (at most two per list)
// recorded candidates with a filter score within 2 eps of the best — those are re-scored with the canonical distance, ties to
// the lowest id — or lies under a list's third-best bound; the same certificate as finalize_kernel then shows the bound cannot
// reach the exact winner. Points that fail it go on to the general pipeline (hard_ids).
__global__ void km_rescore_known_kernel(const void* pts, int dtype, int d, const float* cent, const float* cand_score, const int32_t* cand_id,
                                        const float* cand_thr, int n_lists, int list_len, const float* pnorm2, const float* max_norm_dev,
                                        float rel_eps, float abs_eps, const int32_t* flag_local, const int32_t* flag_count, int64_t base, int64_t* assign,
                                        int64_t* hard_ids, int32_t* hard_count) {
    extern __shared__ __align__(16) float rk_q[];  // [warps per block][d4]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int d4 = ((d + 3) >> 2) << 2;
    float* q_s = rk_q + (size_t)wib * d4;
    const bool vec = (d % 4) == 0;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t nflag = *flag_count;
    const double mx = (double)__ldg(max_norm_dev);
    for (int64_t j = warp; j < nflag; j += nwarps) {
        const int64_t i = flag_local[j];
        const int64_t gi = base + i;
        float f = -INFINITY, thr = -INFINITY;
        int32_t id = -1;
        if (lane < 2 * n_lists) {
            const size_t off = ((size_t)i * n_lists + (lane >> 1)) * list_len + (lane & 1);
            id = cand_id[off];
            if (id >= 0) f = cand_score[off];
        }
        if (lane < n_lists) thr = cand_thr[(size_t)i * n_lists + lane];
        float f1 = f;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            f1 = fmaxf(f1, __shfl_xor_sync(FULL, f1, off));
            thr = fmaxf(thr, __shfl_xor_sync(FULL, thr, off));
        }
        const double qn2 = (double)pnorm2[gi];
        const double qn = sqrt(qn2);
        const double eps_s = 2.0 * filter_ip_err((double)rel_eps, (double)abs_eps, qn, mx) + 2.4e-7 * (mx * mx + 2.0 * qn * mx) + 1.3e-7 * qn2 + 1e-30;
        const double slack = 2.4e-7 * (qn2 + fabs((double)f1));
        const bool contender = id >= 0 && (double)f >= (double)f1 - 2.0 * eps_s - slack;
        // recorded candidates that are not contenders count as discarded rows: fold them into the bound
        float other = (id >= 0 && !contender) ? f : -INFINITY;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) other = fmaxf(other, __shfl_xor_sync(FULL, other, off));
        const float bound = fmaxf(thr, other);
        unsigned todo = __ballot_sync(FULL, contender);
        __syncwarp();
        for (int t = lane; t < d4; t += 32) q_s[t] = t < d ? elem_f32(pts, dtype, (size_t)gi * d + t) : 0.f;
        __syncwarp();
        float best_d = INFINITY;
        int32_t best_c = -1;
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const int32_t c = __shfl_sync(FULL, id, src);
            const double part = canonical_partial<true>(q_s, cent + (size_t)c * d, B2_F32, d, vec, lane);
            const float dist = (float)butterfly_sum(part);
            if (dist < best_d || (dist == best_d && c < best_c)) {
                best_d = dist;
                best_c = c;
            }
        }
        bool ok = best_c >= 0 && best_d == best_d;
        if (ok && bound > -INFINITY) ok = (qn2 * (1.0 - 1.3e-7) - (double)bound - eps_s) > (double)best_d * (1.0 + 2.4e-7) + 1e-30;
        if (lane == 0) {
            if (ok) assign[gi] = best_c;
            else hard_ids[atomicAdd(hard_count, 1)] = gi;
        }
    }
}

__global__ void km_forward_flags_kernel(const int32_t* flag_local, const int32_t* flag_count, int64_t base, int64_t* hard_ids, int32_t* hard_count) {
    const int64_t n = *flag_count;
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x)
        hard_ids[atomicAdd(hard_count, 1)] = base + flag_local[j];
}

__global__ void km_scatter_kernel(const int64_t* flag_ids, int64_t n, const int64_t* sub_assign, int64_t* assign) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j < n) assign[flag_ids[j]] = sub_assign[j];
}

// ---- step 5a: stable counting sort of points by centroid (member lists in point order) --------------------------------
// block b (ONE warp) owns the contiguous point range [b*L, (b+1)*L)
__global__ void km_count_kernel(const int64_t* assign, int64_t n, int64_t L, int k, int32_t* cnt) {
    extern __shared__ int32_t s_cnt[];
    for (int c = threadIdx.x; c < k; c += 32) s_cnt[c] = 0;
    __syncwarp();
    const int64_t lo = blockIdx.x * L, hi = min(n, lo + L);
    for (int64_t i = lo + threadIdx.x; i < hi; i += 32) atomicAdd(&s_cnt[(int)assign[i]], 1);
    __syncwarp();
    for (int c = threadIdx.x; c < k; c += 32) cnt[(size_t)c * gridDim.x + blockIdx.x] = s_cnt[c];  // [k][nb]
}

// per centroid (one warp each): exclusive scan of its nb block counts cnt[c][0..nb); totals[c] = cluster size
__global__ void km_scan_blocks_kernel(int32_t* cnt, int nb, int k, int32_t* totals) {
    const int lane = threadIdx.x & 31;
    const int c = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
    if (c >= k) return;
    int32_t* row = cnt + (size_t)c * nb;
    int32_t run = 0;
    for (int b0 = 0; b0 < nb; b0 += 32) {
        const int b = b0 + lane;
        const int32_t v = b < nb ? row[b] : 0;
        int32_t incl = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int32_t o = __shfl_up_sync(FULL, incl, off);
            if (lane >= off) incl += o;
        }
        if (b < nb) row[b] = run + incl - v;
        run += __shfl_sync(FULL, incl, 31);
    }
    if (lane == 0) totals[c] = run;
}

// offsets[c] = sum of totals[0..c): one block, warp-shuffle scan over chunks of 1024 centroids
__global__ void km_scan_totals_kernel(const int32_t* totals, int k, int64_t* offsets) {
    __shared__ int64_t s_warp[32];
    __shared__ int64_t s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int c0 = 0; c0 < k; c0 += 1024) {
        const int c = c0 + threadIdx.x;
        const int64_t v = c < k ? (int64_t)totals[c] : 0;
        int64_t incl = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int64_t o = __shfl_up_sync(FULL, incl, off);
            if (lane >= off) incl += o;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int64_t before = s_carry;
        for (int w = 0; w < warp; ++w) before += s_warp[w];
        if (c < k) offsets[c] = before + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) offsets[k] = s_carry;
}

__global__ void km_fill_kernel(const int64_t* assign, int64_t n, int64_t L, int k, const int32_t* blk_start, const int64_t* offsets,
                               int32_t* members) {
    extern __shared__ int32_t s_run[];  // next free slot (relative to the cluster's list) for this block's points
    const int lane = threadIdx.x;
    for (int c = lane; c < k; c += 32) s_run[c] = blk_start[(size_t)c * gridDim.x + blockIdx.x];
    __syncwarp();
    const int64_t lo = blockIdx.x * L, hi = min(n, lo + L);
    for (int64_t base = lo; base < hi; base += 32) {
        const int64_t i = base + lane;
        const bool active = i < hi;
        const unsigned amask = __ballot_sync(FULL, active);
        if (active) {
            const int a = (int)assign[i];
            const unsigned same = __match_any_sync(amask, a);
            const int rank = __popc(same & ((1u << lane) - 1));
            const int32_t slot = s_run[a] + rank;
            members[offsets[a] + slot] = (int32_t)i;
            __syncwarp(amask);
            if (rank == 0) s_run[a] += __popc(same);
        }
        __syncwarp();
    }
}

// ---- step 5b: centroid sums in point order ---------------------------------------------------------------------------------
// Every column of a centroid is ONE sequential fp32 chain over its members in point order — that is what makes the centroids
// bit-identical to faiss's compute_centroids — so the adds of a chain cannot be parallelised. What can:
//   * different centroids and different COLUMN chunks are independent: a work item is (centroid, chunk of 32 x V columns),
//     handled by one warp (lane = V consecutive columns = one 16-byte slice of every member row);
//   * the LOADS of a chain: each warp streams its slice of the member rows through a private shared-memory ring with cp.async
//     (ACC_GROUPS x ACC_ROWS = 32 rows in flight, member ids fetched two groups ahead), the dependent adds run over rows that
//     have already landed;
//   * balance: cluster sizes are far from equal while Lloyd is converging (some centroids hold 4x the mean), and the longest
//     chain bounds the pass — warps pull items off a device counter in DECREASING cluster size (km_order_kernel).
// History (profiles/r2_kmeans_accumulate_variants.txt, all at 5M x 768 bf16, k = 1024, one pass):
//   r1  thread per (centroid, column), 2-byte loads ................................ 9.4 ms
//   v1  block per centroid, 16 row loads per lane in registers ..................... 5.3 ms  (DRAM 18 %, SMs busy 29 % of the time)
//   v2  same shape, cp.async ring of 32 rows per block ............................. 6.6 ms  (the per-centroid chain, not load depth, bounds it)
//   v3/v4  warp per (centroid, 512 B chunk), largest cluster first, 32 / 96-row rings  7.4 / 5.5 ms
//   v5  + per-column objective partials (one fp32 chain over a group's 64 products was the critical path), 32-bit ids,
//       unpredicated full groups, 6 warps x 64-row rings per SM .................... 3.6 ms   <- this kernel
//   also tried: 4- and 8-byte lanes (4x / 2x as many, thinner chains), 256-row rings, branch-free predicated copies, TMA bulk
//   copies (cp.async.bulk + mbarrier, one copy per row slice): 3.6-5.0 ms, none better. Per-item counters (B2_KM_DEBUG=1) show
//   why: the largest cluster holds ~48k of the 5M rows (10x the mean) and its chain advances at 110-170 cycles per row whatever
//   the variant, so the pass cannot end before ~48k x 140 cycles = 3.5 ms; the other 3071 items finish long before.
// With OBJ the same pass accumulates sum_members ||x - c_old||^2 (fp32 partials per group, summed in fp64: fp64 issue is scarce).
constexpr int ACC_ROWS = 8;     // rows per cp.async group
constexpr int ACC_SMEM = 192 * 1024;  // ring memory per SM; a warp's ring is NG groups x ACC_ROWS x 32 lanes x LB bytes

// predicated, branch-free: a branch around every copy serialises the eight row copies of a group behind each other's shuffle
template <int LB>
__device__ __forceinline__ void cp_async_lane(void* smem_dst, const void* gsrc, bool pred) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_dst);
    if constexpr (LB == 16)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p cp.async.cg.shared.global [%0], [%1], 16;\n\t}" ::"r"(dst), "l"(gsrc), "r"((int)pred) : "memory");
    else if constexpr (LB == 8)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p cp.async.ca.shared.global [%0], [%1], 8;\n\t}" ::"r"(dst), "l"(gsrc), "r"((int)pred) : "memory");
    else
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p cp.async.ca.shared.global [%0], [%1], 4;\n\t}" ::"r"(dst), "l"(gsrc), "r"((int)pred) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// order[i] = centroid ids by decreasing size class (floor(log2(size)); exact order inside a class does not matter): one block
__global__ void km_order_kernel(const int32_t* totals, int k, int32_t* order) {
    __shared__ int s_cnt[33], s_base[33];
    if (threadIdx.x < 33) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (int c = threadIdx.x; c < k; c += blockDim.x) atomicAdd(&s_cnt[32 - __clz(max(totals[c], 0))], 1);  // class 0: empty
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int cls = 32; cls >= 0; --cls) {
            s_base[cls] = run;
            run += s_cnt[cls];
        }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < k; c += blockDim.x) order[atomicAdd(&s_base[32 - __clz(max(totals[c], 0))], 1)] = c;
}

template <int LB> struct LaneWord;
template <> struct LaneWord<16> { using T = uint4; };
template <> struct LaneWord<8> { using T = uint2; };
template <> struct LaneWord<4> { using T = uint32_t; };

// LB = bytes of a member row per lane (4, 8 or 16): a warp covers 32 * LB contiguous bytes of every member row. Small LB = more,
// shorter-per-row chains: the time of the pass is bounded below by (largest cluster) x (cycles per row of ONE warp), and the
// largest cluster is ~10x the mean while Lloyd converges on the benchmark mixture (48k of 5M rows at k = 1024).
template <int DT, bool OBJ, int LB, int ACC_GROUPS>  // DT: element type of the rows (B2_F32, B2_BF16 or B2_F16)
__global__ void __launch_bounds__(256) km_accumulate_vec_kernel(const void* x, int d, const int64_t* ids, const int32_t* members,
                                                                const int64_t* offsets, const int32_t* order, const float* cent_old,
                                                                float* cent_out, float* hassign, double* obj, int normalize, int k,
                                                                int n_chunks, int* work_counter, long long* dbg) {
    constexpr int V = DT != B2_F32 ? LB / 2 : LB / 4;  // columns per lane
    using Word = typename LaneWord<LB>::T;
    extern __shared__ __align__(16) uint8_t acc_ring_raw[];  // [warps][ACC_GROUPS * ACC_ROWS][32] words
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    Word* my_ring = reinterpret_cast<Word*>(acc_ring_raw) + (size_t)wib * (ACC_GROUPS * ACC_ROWS * 32) + lane;
    const size_t row_bytes = (size_t)d * (DT != B2_F32 ? 2 : 4);
    const int row_words = (int)(row_bytes / LB);
    const int n_items = k * n_chunks;
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(work_counter, 1);
        item = __shfl_sync(FULL, item, 0);
        if (item >= n_items) break;
        const long long dbg_t0 = dbg ? clock64() : 0;
        const int c = order[item / n_chunks];
        const int chunk = item - (item / n_chunks) * n_chunks;
        const int word = chunk * 32 + lane;  // this lane's LB-byte slice inside a row
        const int col0 = word * V;
        const bool active = word < row_words;
        const int64_t o0 = offsets[c], o1 = offsets[c + 1];
        const int64_t nmem = o1 - o0;
        const float cntf = (float)nmem;
        if (chunk == 0 && lane == 0) hassign[c] = cntf;
        float acc[V], cold[V], part[V];  // sums, old centroid (objective), objective partials (one chain per column)
#pragma unroll
        for (int j = 0; j < V; ++j) {
            acc[j] = 0.f;
            part[j] = 0.f;
            cold[j] = (OBJ && active) ? cent_old[(size_t)c * d + col0 + j] : 0.f;
        }
        double dsum = 0.0;
        const int64_t ngroups = (nmem + ACC_ROWS - 1) / ACC_ROWS;
        // member rows are fetched 32 at a time (one coalesced load = 4 groups), three such batches ahead of the issue point
        constexpr int GPB = 32 / ACC_ROWS;  // groups per id batch
        auto fetch_batch = [&](int64_t b) -> int32_t {  // lane l: member row (b * 32 + l) of this centroid, -1 past the end
            const int64_t o = o0 + b * 32 + lane;
            if (o >= o1) return -1;
            const int32_t p = members[o];
            return ids ? (int32_t)ids[p] : p;  // row numbers fit 32 bits (the filter's ids are 32-bit too)
        };
        const char* xb = reinterpret_cast<const char*>(x) + (size_t)word * LB;
        auto issue = [&](int64_t g, int32_t batch_ids) {  // all lanes call it; row u of group g sits in lane (g % GPB) * ACC_ROWS + u
            Word* dst = my_ring + (size_t)((int)(g % ACC_GROUPS) * ACC_ROWS) * 32;
            const int lane0 = (int)(g % GPB) * ACC_ROWS;
            int32_t r[ACC_ROWS];
#pragma unroll
            for (int u = 0; u < ACC_ROWS; ++u) r[u] = __shfl_sync(FULL, batch_ids, lane0 + u);
#pragma unroll
            for (int u = 0; u < ACC_ROWS; ++u)
                cp_async_lane<LB>(dst + u * 32, xb + (size_t)(uint32_t)max(r[u], 0) * row_bytes, r[u] >= 0 && active);
            cp_async_commit();
        };
        auto consume_row = [&](const Word& raw) {
            float v[V];
            const uint32_t* w32 = reinterpret_cast<const uint32_t*>(&raw);
            if constexpr (DT == B2_F16) {
#pragma unroll
                for (int t = 0; t < LB / 4; ++t) {
                    const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&w32[t]));
                    v[2 * t] = h.x;
                    v[2 * t + 1] = h.y;
                }
            } else if constexpr (DT == B2_BF16) {
#pragma unroll
                for (int t = 0; t < LB / 4; ++t) {
                    v[2 * t] = __uint_as_float(w32[t] << 16);
                    v[2 * t + 1] = __uint_as_float(w32[t] & 0xffff0000u);
                }
            } else {
#pragma unroll
                for (int t = 0; t < LB / 4; ++t) v[t] = __uint_as_float(w32[t]);
            }
#pragma unroll
            for (int j = 0; j < V; ++j) acc[j] = __fadd_rn(acc[j], v[j]);
            if constexpr (OBJ) {
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const float df = v[j] - cold[j];
                    part[j] = fmaf(df, df, part[j]);
                }
            }
        };
        // prologue: ACC_GROUPS groups in flight (ACC_GROUPS / GPB id batches), then three batches of ids in registers
        static_assert(ACC_GROUPS % GPB == 0, "the prologue issues whole id batches");
        for (int b = 0; b < ACC_GROUPS / GPB; ++b) {
            const int32_t bi = fetch_batch(b);
            for (int gg = 0; gg < GPB; ++gg) issue((int64_t)b * GPB + gg, bi);
        }
        int32_t ids_a = fetch_batch(ACC_GROUPS / GPB), ids_b = fetch_batch(ACC_GROUPS / GPB + 1), ids_c = fetch_batch(ACC_GROUPS / GPB + 2);
        for (int64_t g = 0; g < ngroups; ++g) {
            cp_async_wait<ACC_GROUPS - 1>();  // group g has landed (the groups behind it may still be in flight)
            const Word* src = my_ring + (size_t)((int)(g % ACC_GROUPS) * ACC_ROWS) * 32;
            const int nrows = (int)((nmem - g * ACC_ROWS) < ACC_ROWS ? (nmem - g * ACC_ROWS) : ACC_ROWS);
            if (active) {
                if (nrows == ACC_ROWS) {
#pragma unroll
                    for (int u = 0; u < ACC_ROWS; ++u) consume_row(src[u * 32]);
                } else {
                    for (int u = 0; u < nrows; ++u) consume_row(src[u * 32]);
                }
            }
            if constexpr (OBJ) {
                if ((g & 7) == 7 || g + 1 == ngroups) {  // fold the fp32 partials into the fp64 total every 64 rows
                    float t = 0.f;
#pragma unroll
                    for (int j = 0; j < V; ++j) {
                        t += part[j];
                        part[j] = 0.f;
                    }
                    dsum += (double)t;
                }
            }
            __syncwarp();
            // refill the slot just consumed with group g + ACC_GROUPS (its ids are in ids_a); rotate the id batches every GPB groups
            const int64_t gi = g + ACC_GROUPS;
            issue(gi, ids_a);
            if ((gi % GPB) == GPB - 1) {
                ids_a = ids_b;
                ids_b = ids_c;
                ids_c = fetch_batch(gi / GPB + 3);
            }
        }
        cp_async_wait<0>();
        if (active) {
            float norm = 1.f;
            if (normalize && nmem > 0) norm = __fdiv_rn(1.0f, cntf);
#pragma unroll
            for (int j = 0; j < V; ++j) cent_out[(size_t)c * d + col0 + j] = (normalize && nmem > 0) ? __fmul_rn(acc[j], norm) : acc[j];
        }
        if constexpr (OBJ) {
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) dsum += __shfl_xor_sync(FULL, dsum, off);
            if (lane == 0 && dsum != 0.0) atomicAdd(obj, dsum);
        }
        if (dbg && lane == 0) {  // B2_KM_DEBUG: (rows, cycles, start clock, SM) of every work item
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            dbg[4 * (size_t)item + 0] = nmem;
            dbg[4 * (size_t)item + 1] = clock64() - dbg_t0;
            dbg[4 * (size_t)item + 2] = dbg_t0;
            dbg[4 * (size_t)item + 3] = smid;
        }
        __syncwarp();
    }
}

// generic shapes (row size not a multiple of 16 bytes): thread (c, j) sums column j over the members in point order
__global__ void km_accumulate_kernel(const void* x, int dtype, int d, const int64_t* ids, const int32_t* members,
                                     const int64_t* offsets, const float* cent_old, float* cent_out, float* hassign, double* obj,
                                     int normalize) {
    const int c = blockIdx.x;
    const int64_t o0 = offsets[c], o1 = offsets[c + 1];
    const float cntf = (float)(o1 - o0);
    if (threadIdx.x == 0 && blockIdx.y == 0) hassign[c] = cntf;
    const int j = blockIdx.y * blockDim.x + threadIdx.x;
    const bool active = j < d;
    float acc = 0.f;
    double dsum = 0.0;
    const float cold = (cent_old && active) ? cent_old[(size_t)c * d + j] : 0.f;
    if (active) {
        for (int64_t o = o0; o < o1; ++o) {
            const int64_t p = members[o];
            const int64_t r = ids ? ids[p] : p;
            const float v = elem_f32(x, dtype, (size_t)(r * d + j));
            acc = __fadd_rn(acc, v);
            if (cent_old) {
                const float df = v - cold;
                dsum += (double)(df * df);
            }
        }
        if (normalize && o1 > o0) acc = __fmul_rn(acc, __fdiv_rn(1.0f, cntf));
        cent_out[(size_t)c * d + j] = acc;
    }
    if (cent_old) {
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) dsum += __shfl_xor_sync(FULL, dsum, off);
        if ((threadIdx.x & 31) == 0 && dsum != 0.0) atomicAdd(obj, dsum);
    }
}

// ---- step 6: faiss/Clustering.cpp split_clusters (EPS = 1/1024, RandomGenerator rng(1234) = std::mt19937) on the device ----
// One block. Clusters are visited in order; an empty one takes a copy of a cluster cj drawn with probability proportional to
// its size (rejection loop over cj = 0, 1, ... with rng.rand_float() = mt() / float(mt.max())), the two copies are perturbed
// symmetrically and the size is shared. The draws depend on the sizes left by earlier splits, so the walk is sequential;
// thread 0 draws, the block copies.
// The draws depend on the sizes left by earlier splits, so clusters are visited sequentially; WITHIN one visit the rejection walk
// is parallel: the 624 outputs of an MT19937 state are produced by the whole block (the twist in three dependent phases), every
// thread tests one (draw, candidate) pair of the walk, and the first acceptance in walk order wins (block-wide minimum).
__device__ __forceinline__ uint32_t mt_mix(uint32_t a, uint32_t b) {
    const uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
    return (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}
__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

__global__ void __launch_bounds__(256) km_split_kernel(int d, int k, int64_t n, float* hassign, float* centroids) {
    __shared__ uint32_t s_mt[624], s_old[624];
    __shared__ float s_r[624];  // rng.rand_float() = mt() / float(mt.max()) of the current state's outputs
    __shared__ int s_pos, s_found;
    const int tid = threadIdx.x;
    int any = 0;
    for (int c = tid; c < k; c += blockDim.x) any |= hassign[c] == 0.f;
    if (!__syncthreads_or(any)) return;
    if (tid == 0) {  // std::mt19937(1234)
        s_mt[0] = 1234u;
        for (int i = 1; i < 624; ++i) s_mt[i] = 1812433253u * (s_mt[i - 1] ^ (s_mt[i - 1] >> 30)) + (uint32_t)i;
        s_pos = 624;  // no output generated yet
    }
    __syncthreads();
    const double EPS = 1 / 1024.;
    const double denom = (double)(float)(n - k);
    for (int ci = 0; ci < k; ++ci) {
        if (hassign[ci] != 0.f) continue;  // block-uniform (sizes are only written between barriers)
        // for (cj = 0; true; cj = (cj + 1) % k) { p = (hassign[cj] - 1.0) / (float)(n - k); r = rng.rand_float(); if (r < p) break; }
        int64_t tries = 0;
        int cj = 0;
        for (;;) {
            if (s_pos >= 624) {  // next state: mt[i] = mt[i+397 mod 624] ^ mix(mt[i], mt[i+1]) with already-updated sources for i >= 227
                for (int i = tid; i < 624; i += blockDim.x) s_old[i] = s_mt[i];
                __syncthreads();
                for (int i = tid; i < 227; i += blockDim.x) s_mt[i] = s_old[i + 397] ^ mt_mix(s_old[i], s_old[i + 1]);
                __syncthreads();
                for (int i = 227 + tid; i < 454; i += blockDim.x) s_mt[i] = s_mt[i - 227] ^ mt_mix(s_old[i], s_old[i + 1]);
                __syncthreads();
                for (int i = 454 + tid; i < 623; i += blockDim.x) s_mt[i] = s_mt[i - 227] ^ mt_mix(s_old[i], s_old[i + 1]);
                __syncthreads();
                if (tid == 0) {
                    s_mt[623] = s_mt[396] ^ mt_mix(s_old[623], s_mt[0]);
                    s_pos = 0;
                }
                __syncthreads();
                for (int i = tid; i < 624; i += blockDim.x) s_r[i] = __fdiv_rn(__uint2float_rn(mt_temper(s_mt[i])), 4294967296.0f);
                __syncthreads();
            }
            const int pos = s_pos, avail = 624 - pos;
            if (tid == 0) s_found = 0x7fffffff;
            __syncthreads();
            for (int j = tid; j < avail; j += blockDim.x) {
                const int c = (int)((tries + j) % k);
                const float p = (float)(((double)hassign[c] - 1.0) / denom);
                if (s_r[pos + j] < p) atomicMin(&s_found, j);
            }
            __syncthreads();
            const int f = s_found;
            __syncthreads();
            if (f != 0x7fffffff) {
                cj = (int)((tries + f) % k);
                if (tid == 0) s_pos = pos + f + 1;
                __syncthreads();
                break;
            }
            tries += avail;
            if (tid == 0) s_pos = 624;
            __syncthreads();
        }
        for (int j = tid; j < d; j += blockDim.x) {
            const float src = centroids[(size_t)cj * d + j];
            const double up = 1 + EPS, down = 1 - EPS;
            centroids[(size_t)ci * d + j] = (float)((double)src * ((j % 2 == 0) ? up : down));
            centroids[(size_t)cj * d + j] = (float)((double)src * ((j % 2 == 0) ? down : up));
        }
        __syncthreads();
        if (tid == 0) {
            const float hv = hassign[cj] / 2;
            hassign[ci] = hv;
            hassign[cj] -= hv;
        }
        __syncthreads();
    }
}

// searchable view of the fp32 centroid matrix; the filter operand matches the point dtype (bf16 / fp16 points -> a bf16 / fp16
// copy; the fp16 rounding of the centroids is in the certificate through filter_rel_eps / filter_abs_eps).
// No host synchronisation: the max norm stays in device memory (MatView::max_norm_dev).
int centroid_view(const float* cent, int k, int d, int point_dtype, KmWork& w, MatView& v, cudaStream_t st) {
    v.store = cent;
    v.n = k;
    v.d = d;
    v.dtype = B2_F32;
    if (point_dtype == B2_BF16 || point_dtype == B2_F16) {
        v.filt_dtype = point_dtype;
        v.filt_pitch = round_up(d, 8);
        B2_TRY(w.cent_filt.ensure((size_t)k * v.filt_pitch * 2));
        B2_TRY(w.scalar.ensure(64));
        int32_t* overflow = reinterpret_cast<int32_t*>(w.scalar.as<char>() + 32);  // read back by assign_points
        B2_CUDA(cudaMemsetAsync(overflow, 0, sizeof(int32_t), st));
        B2_TRY(launch_convert_pad(cent, B2_F32, k, d, w.cent_filt.p, point_dtype, v.filt_pitch, st, overflow));
        v.filt = w.cent_filt.p;
    } else {
        v.filt_dtype = B2_F32;
        if (d % 4 == 0) {
            v.filt = cent;
            v.filt_pitch = d;
        } else {
            v.filt_pitch = round_up(d, 4);
            B2_TRY(w.cent_filt.ensure((size_t)k * v.filt_pitch * 4));
            B2_TRY(launch_convert_pad(cent, B2_F32, k, d, w.cent_filt.p, B2_F32, v.filt_pitch, st));
            v.filt = w.cent_filt.p;
        }
    }
    B2_TRY(w.cent_norm2.ensure((size_t)k * sizeof(float)));
    B2_TRY(w.scalar.ensure(64));
    B2_TRY(launch_row_norms(cent, B2_F32, k, d, w.cent_norm2.as<float>(), w.scalar.as<float>(), st));
    v.norm2 = w.cent_norm2.as<float>();
    v.max_norm = 0.f;
    v.max_norm_dev = w.scalar.as<float>();
    return B2_OK;
}

// assign[m] (int64, device) for the rows pts[m,d] (device, index dtype; pnorm2[m] = their canonical squared norms) against
// the k centroids cent[k,d] (fp32, device). Steps 1-4 of the header.
int assign_points(b2_index* idx, const void* pts, const float* pnorm2, int64_t m, const float* cent, int k, KmWork& w, int64_t* assign,
                  cudaStream_t st, int64_t* n_second_level = nullptr) {
    idx->last_filter_ms = -1.f;
    if (n_second_level) *n_second_level = 0;
    if (m <= 0) return B2_OK;
    const int d = idx->d;
    MatView cv;
    B2_TRY(centroid_view(cent, k, d, idx->dtype, w, cv, st));
    int dev_sms = 148;
    cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, idx->device);
    const int filt_dtype = cv.filt_dtype;
    const int kp = 16;
    const int64_t q_pitch = round_up(d, filt_dtype == B2_F32 ? 4 : 8);
    const float rel_eps = filter_rel_eps(B2_F32, filt_dtype, idx->dtype, d);
    const float abs_eps = filter_abs_eps(B2_F32, filt_dtype, idx->dtype, d);
    const bool q_in_place = idx->dtype == filt_dtype && q_pitch == d && (reinterpret_cast<uintptr_t>(pts) & 15) == 0;
    const int64_t chunk = (int64_t)1 << 23;
    B2_TRY(w.flag_ids.ensure((size_t)std::min(m, chunk) * sizeof(int32_t)));
    B2_TRY(w.hard_ids.ensure((size_t)m * sizeof(int64_t)));
    B2_TRY(w.flag_count.ensure(64));
    B2_TRY(w.h_count.ensure(64));
    int32_t* flag_count = w.flag_count.as<int32_t>();
    int32_t* hard_count = flag_count + 1;
    B2_CUDA(cudaMemsetAsync(flag_count, 0, 2 * sizeof(int32_t), st));
    const int d4 = ((d + 3) >> 2) << 2;
    const size_t rk_smem = (size_t)8 * d4 * sizeof(float);
    if (rk_smem > 200 * 1024) {
        set_error("embedding dimension %d too large for the k-means re-score kernel", d);
        return B2_ERANGE;
    }
    if (rk_smem > 48 * 1024) B2_CUDA(cudaFuncSetAttribute(km_rescore_known_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rk_smem));
    B2_CUDA(cudaEventRecord(idx->ev0, st));
    for (int64_t q0 = 0; q0 < m; q0 += chunk) {
        const int64_t mc = std::min<int64_t>(chunk, m - q0);
        const char* pc = reinterpret_cast<const char*>(pts) + (size_t)q0 * d * esize(idx->dtype);
        const bool two_cta = filter_use_pair(mc);
        const int n_splits = filter_choose_splits(mc, k, dev_sms, two_cta, /*top1=*/true);
        if (!q_in_place) {
            B2_TRY(idx->q_filt.ensure((size_t)mc * q_pitch * esize(filt_dtype)));
            B2_TRY(launch_prep_queries(pc, idx->dtype, mc, d, idx->q_filt.p, filt_dtype, q_pitch, st));
        }
        const void* q_filt = q_in_place ? static_cast<const void*>(pc) : idx->q_filt.p;
        B2_TRY(idx->cand_score.ensure((size_t)mc * n_splits * kp * sizeof(float)));
        B2_TRY(idx->cand_id.ensure((size_t)mc * n_splits * kp * sizeof(int32_t)));
        B2_TRY(idx->cand_thr.ensure((size_t)mc * n_splits * 2 * sizeof(float)));
        B2_TRY(launch_knn_filter(cv, q_filt, q_pitch, mc, B2_METRIC_L2, kp, n_splits, two_cta, idx->cand_score.as<float>(),
                                 idx->cand_id.as<int32_t>(), idx->cand_thr.as<float>(), idx->device, st, /*top1=*/true));
        if (q0 + chunk >= m) B2_CUDA(cudaEventRecord(idx->ev1, st));
        if (q0 > 0) B2_CUDA(cudaMemsetAsync(flag_count, 0, sizeof(int32_t), st));
        km_assign_finalize_kernel<<<(unsigned)ceil_div(mc, 256), 256, 0, st>>>(
            idx->cand_score.as<float>(), idx->cand_id.as<int32_t>(), idx->cand_thr.as<float>(), mc, 2 * n_splits, kp / 2, pnorm2,
            cv.max_norm_dev, rel_eps, abs_eps, assign, w.flag_ids.as<int32_t>(), flag_count, q0);
        B2_LAUNCH_CHECK();
        // the flagged points of this chunk, while its candidate lists are still in the workspace (count read on the device)
        if (4 * n_splits <= 32)
            km_rescore_known_kernel<<<dev_sms * 4, 256, rk_smem, st>>>(pts, idx->dtype, d, cent, idx->cand_score.as<float>(),
                                                                     idx->cand_id.as<int32_t>(), idx->cand_thr.as<float>(), 2 * n_splits, kp / 2,
                                                                     pnorm2, cv.max_norm_dev, rel_eps, abs_eps, w.flag_ids.as<int32_t>(), flag_count, q0,
                                                                     assign, w.hard_ids.as<int64_t>(), hard_count);
        else
            km_forward_flags_kernel<<<dev_sms, 256, 0, st>>>(w.flag_ids.as<int32_t>(), flag_count, q0, w.hard_ids.as<int64_t>(), hard_count);
        B2_LAUNCH_CHECK();
    }
    int32_t* h_count = reinterpret_cast<int32_t*>(w.h_count.p);
    B2_CUDA(cudaMemcpyAsync(h_count, hard_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    h_count[1] = 0;
    if (filt_dtype == B2_F16) B2_CUDA(cudaMemcpyAsync(h_count + 1, w.scalar.as<char>() + 32, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    cudaError_t se = cudaStreamSynchronize(st);
    if (se != cudaSuccess) {
        set_error("k-means assignment failed on the device: %s", cudaGetErrorString(se));
        return B2_ECUDA;
    }
    if (h_count[1]) {  // the fp16 filter copy of a centroid would not be finite: no certificate can hold
        set_error("a k-means centroid has an element beyond the fp16 range (|x| >= 65520) of this fp16 store");
        return B2_ERANGE;
    }
    float ms = -1.f;
    if (cudaEventElapsedTime(&ms, idx->ev0, idx->ev1) == cudaSuccess) idx->last_filter_ms = ms;
    const int64_t nf = *h_count;
    g_stats[ST_QUERIES] += m - nf;  // (search_core counts the hard points itself)
    if (n_second_level) *n_second_level = nf;
    if (nf > 0) {
        // points neither the gap test nor the known-contender certificate could settle (exact ties across lists, near-ties
        // with undiscovered centroids): the general exact pipeline on the gathered rows
        const float filt_ms = idx->last_filter_ms;
        B2_TRY(w.sub.ensure((size_t)nf * d * esize(idx->dtype)));
        B2_TRY(w.sub_dis.ensure((size_t)nf * sizeof(float)));
        B2_TRY(w.sub_assign.ensure((size_t)nf * sizeof(int64_t)));
        int* err = reinterpret_cast<int*>(w.scalar.as<char>() + 16);
        B2_TRY(launch_gather_rows(pts, idx->dtype, d, w.hard_ids.as<int64_t>(), nf, m, w.sub.p, err, st));
        B2_TRY(search_core(idx, cv, B2_METRIC_L2, w.sub.p, idx->dtype, nf, 1, nullptr, 0, w.sub_dis.as<float>(), w.sub_assign.as<int64_t>(), st));
        km_scatter_kernel<<<(unsigned)ceil_div(nf, 256), 256, 0, st>>>(w.hard_ids.as<int64_t>(), nf, w.sub_assign.as<int64_t>(), assign);
        B2_LAUNCH_CHECK();
        idx->last_filter_ms = filt_ms;
    }
    return B2_OK;
}

// Steps 5-6: member lists, centroid sums (into cent_out), optional objective against cent_old, optional split.
int update_centroids(b2_index* idx, const void* x, const int64_t* row_ids, int64_t n, const int64_t* assign, int k, KmWork& w,
                     const float* cent_old, float* cent_out, double* obj, cudaStream_t st, int normalize) {
    const int d = idx->d;
    // one warp per block walks its point range in order; <= 1024 ranges keep the per-centroid scan over blocks short
    int64_t nb = std::min<int64_t>(1024, std::max<int64_t>(1, ceil_div(n, 256)));
    while (nb > 1 && nb * (int64_t)k > ((int64_t)1 << 26)) nb /= 2;
    const int64_t L = ceil_div(std::max<int64_t>(n, 1), nb);
    nb = std::max<int64_t>(1, ceil_div(n, L));
    const size_t smem = (size_t)k * sizeof(int32_t);
    if (smem > 200 * 1024) {
        set_error("k=%d centroids exceed the shared-memory budget of the member-list kernels", k);
        return B2_ERANGE;
    }
    if (smem > 48 * 1024) {
        B2_CUDA(cudaFuncSetAttribute(km_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        B2_CUDA(cudaFuncSetAttribute(km_fill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    B2_TRY(w.blk.ensure((size_t)nb * k * sizeof(int32_t)));
    B2_TRY(w.totals.ensure((size_t)k * sizeof(int32_t)));
    B2_TRY(w.offsets.ensure((size_t)(k + 1) * sizeof(int64_t)));
    B2_TRY(w.members.ensure((size_t)std::max<int64_t>(n, 1) * sizeof(int32_t)));
    B2_TRY(w.hassign.ensure((size_t)k * sizeof(float)));
    km_count_kernel<<<(unsigned)nb, 32, smem, st>>>(assign, n, L, k, w.blk.as<int32_t>());
    B2_LAUNCH_CHECK();
    km_scan_blocks_kernel<<<(unsigned)ceil_div(k, 8), 256, 0, st>>>(w.blk.as<int32_t>(), (int)nb, k, w.totals.as<int32_t>());
    B2_LAUNCH_CHECK();
    km_scan_totals_kernel<<<1, 1024, 0, st>>>(w.totals.as<int32_t>(), k, w.offsets.as<int64_t>());
    B2_LAUNCH_CHECK();
    km_fill_kernel<<<(unsigned)nb, 32, smem, st>>>(assign, n, L, k, w.blk.as<int32_t>(), w.offsets.as<int64_t>(), w.members.as<int32_t>());
    B2_LAUNCH_CHECK();
    // Bytes of a member row per lane: 16 (a warp covers 512 B of the row, fewest instructions per byte) unless that leaves too few
    // (centroid, chunk) chains to occupy the machine — few centroids — then 4 (128 B per warp, 4x as many chains).
    // B2_KM_LANE_BYTES = 4 | 16 overrides. Measured at 5M x 768, k = 1024 (profiles/r2_kmeans_accumulate_variants.txt): the pass is
    // bounded by the LARGEST cluster's chain (~48k of 5M rows, 10x the mean, while Lloyd converges) at ~110-170 cycles per row of
    // one warp, whatever the lane width (4 / 8 / 16 B), the ring depth (64 / 256 rows) or the copy mechanism (cp.async / TMA bulk).
    static const int lane_bytes_env = [] { const char* e = getenv("B2_KM_LANE_BYTES"); const int v = e ? atoi(e) : 0; return (v == 4 || v == 16) ? v : 0; }();
    const size_t row_bytes_total = (size_t)d * esize(idx->dtype);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, idx->device);
    int LB = lane_bytes_env ? lane_bytes_env : ((int64_t)k * (int64_t)ceil_div((int64_t)row_bytes_total, 512) >= 4LL * 6 * sms ? 16 : 4);
    if (LB == 16 && (row_bytes_total % 16 != 0 || (reinterpret_cast<uintptr_t>(x) % 16) != 0)) LB = 4;
    const bool vec_ok = row_bytes_total % LB == 0 && (reinterpret_cast<uintptr_t>(x) % LB) == 0;
    if (vec_ok) {
        const int n_chunks = (int)ceil_div((int64_t)(row_bytes_total / LB), 32);
        const int NG = LB == 16 ? 8 : 32;  // cp.async groups of 8 rows in flight per warp: a 32 KB ring either way, 6 warps per SM
        const size_t warp_ring = (size_t)NG * ACC_ROWS * 32 * LB;
        const int warps = 2;
        const size_t ring = warp_ring * warps;
        const bool want_obj = cent_old != nullptr;
        B2_TRY(w.scalar.ensure(64));
        B2_TRY(w.order.ensure((size_t)k * sizeof(int32_t)));
        int* counter = reinterpret_cast<int*>(w.scalar.as<char>() + 48);
        B2_CUDA(cudaMemsetAsync(counter, 0, sizeof(int), st));
        km_order_kernel<<<1, 1024, 0, st>>>(w.totals.as<int32_t>(), k, w.order.as<int32_t>());
        B2_LAUNCH_CHECK();
        static const bool dbg_on = [] { const char* e = getenv("B2_KM_DEBUG"); return e && atoi(e) != 0; }();
        long long* dbg = nullptr;
        if (dbg_on) {
            B2_TRY(w.dbg.ensure((size_t)k * n_chunks * 4 * sizeof(long long)));
            dbg = w.dbg.as<long long>();
        }
#define B2_ACC_LAUNCH(BF, OB, LBV, NGV)                                                                                           \
    do {                                                                                                                          \
        auto kern = km_accumulate_vec_kernel<BF, OB, LBV, NGV>;                                                                   \
        B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring));                              \
        int per_sm = 1;                                                                                                           \
        B2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, ring));                                  \
        per_sm = std::max(1, std::min<int>(per_sm, (int)(ACC_SMEM / ring)));                                                      \
        const int grid = (int)std::min<int64_t>(ceil_div((int64_t)k * n_chunks, warps), (int64_t)per_sm * sms);                   \
        kern<<<grid, warps * 32, ring, st>>>(x, d, row_ids, w.members.as<int32_t>(), w.offsets.as<int64_t>(), w.order.as<int32_t>(), \
                                             cent_old, cent_out, w.hassign.as<float>(), obj, normalize, k, n_chunks, counter, dbg); \
    } while (0)
#define B2_ACC_LB(BF, OB)                              \
    do {                                               \
        if (LB == 16) B2_ACC_LAUNCH(BF, OB, 16, 8);    \
        else B2_ACC_LAUNCH(BF, OB, 4, 32);             \
    } while (0)
        if (idx->dtype == B2_BF16) {
            if (want_obj) B2_ACC_LB(B2_BF16, true);
            else B2_ACC_LB(B2_BF16, false);
        } else if (idx->dtype == B2_F16) {
            if (want_obj) B2_ACC_LB(B2_F16, true);
            else B2_ACC_LB(B2_F16, false);
        } else {
            if (want_obj) B2_ACC_LB(B2_F32, true);
            else B2_ACC_LB(B2_F32, false);
        }
#undef B2_ACC_LB
#undef B2_ACC_LAUNCH
        if (dbg) {
            std::vector<long long> h((size_t)k * n_chunks * 4);
            cudaStreamSynchronize(st);
            cudaMemcpy(h.data(), dbg, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
            long long rows_tot = 0;
            size_t worst = 0;
            for (size_t i = 0; i < (size_t)k * n_chunks; ++i) {
                rows_tot += h[4 * i];
                if (h[4 * i + 1] > h[4 * worst + 1]) worst = i;
            }
            fprintf(stderr, "[b2 km accumulate dbg] lane bytes %d, items %d, rows/item mean %.0f | slowest item: %lld rows in %lld cycles (%.0f cycles/row), SM %lld\n",
                    LB, k * n_chunks, (double)rows_tot / (k * n_chunks), h[4 * worst], h[4 * worst + 1],
                    (double)h[4 * worst + 1] / std::max<long long>(h[4 * worst], 1), h[4 * worst + 3]);
        }
    } else {
        dim3 grid((unsigned)k, (unsigned)ceil_div(d, 128));
        km_accumulate_kernel<<<grid, 128, 0, st>>>(x, idx->dtype, d, row_ids, w.members.as<int32_t>(), w.offsets.as<int64_t>(), cent_old,
                                                   cent_out, w.hassign.as<float>(), obj, normalize);
    }
    B2_LAUNCH_CHECK();
    return B2_OK;
}

// B2_KM_TIMING=1: per-phase wall clock of b2_kmeans on stderr (each phase closed by a stream synchronise: a diagnostic, not a
// benchmark mode)
struct KmTimer {
    bool on;
    cudaStream_t st;
    std::chrono::steady_clock::time_point t0;
    double acc[6] = {0, 0, 0, 0, 0, 0};  // setup, assign, assign:filter, update, -, final
    int64_t second_level = 0;
    KmTimer(cudaStream_t s) : st(s) {
        const char* e = getenv("B2_KM_TIMING");
        on = e && atoi(e) != 0;
        t0 = std::chrono::steady_clock::now();
    }
    void lap(int slot) {
        if (!on) return;
        cudaStreamSynchronize(st);
        const auto t1 = std::chrono::steady_clock::now();
        acc[slot] += std::chrono::duration<double, std::milli>(t1 - t0).count();
        t0 = t1;
    }
    void report(int64_t m, int64_t nx, int k, int d, int niter) const {
        if (!on) return;
        fprintf(stderr,
                "[b2 kmeans timing] m=%lld train=%lld k=%d d=%d niter=%d | setup %.2f ms | %d x assign %.2f ms (filter kernel %.2f, "
                "second-level points %lld) | %d x update+split %.2f ms | final assign %.2f ms\n",
                (long long)m, (long long)nx, k, d, niter, acc[0], niter, acc[1], acc[2], (long long)second_level, niter, acc[3], acc[5]);
    }
};

// the point set of a call: all rows of the index, or the rows ids[0..m) gathered into w.pts; norms alongside
int point_set(b2_index* idx, const int64_t* ids_dev, int64_t m, KmWork& w, const void*& P, const float*& Pn, cudaStream_t st) {
    P = idx->store.p;
    Pn = idx->view.norm2;
    if (!ids_dev) return B2_OK;
    const int d = idx->d;
    B2_TRY(w.pts.ensure((size_t)std::max<int64_t>(m, 1) * d * esize(idx->dtype)));
    B2_TRY(w.pts_norm2.ensure((size_t)std::max<int64_t>(m, 1) * sizeof(float)));
    B2_TRY(w.scalar.ensure(64));
    int* err = reinterpret_cast<int*>(w.scalar.as<char>() + 16);
    B2_CUDA(cudaMemsetAsync(err, 0, sizeof(int), st));
    B2_TRY(launch_gather_rows(idx->store.p, idx->dtype, d, ids_dev, m, idx->n, w.pts.p, err, st));
    B2_TRY(launch_row_norms(w.pts.p, idx->dtype, m, d, w.pts_norm2.as<float>(), w.scalar.as<float>() + 8, st));
    int herr = 0;
    B2_CUDA(cudaMemcpyAsync(&herr, err, sizeof(int), cudaMemcpyDeviceToHost, st));
    B2_CUDA(cudaStreamSynchronize(st));
    if (herr) {
        set_error("ids contains a position outside [0, %lld)", (long long)idx->n);
        return B2_ERANGE;
    }
    P = w.pts.p;
    Pn = w.pts_norm2.as<float>();
    return B2_OK;
}

int kmeans_impl(b2_index* idx, const int64_t* ids_host, int64_t m, int k, int niter, int64_t seed, int full_lloyd, int64_t* out_assign,
                float* out_centroids, float* out_obj, KmWork& w) {
    const int d = idx->d;
    cudaStream_t st = idx->stream;
    KmTimer tm(st);
    const size_t es = esize(idx->dtype);
    const int64_t* ids_dev = nullptr;
    if (ids_host) {
        B2_TRY(w.ids.ensure((size_t)std::max<int64_t>(m, 1) * sizeof(int64_t)));
        B2_CUDA(cudaMemcpyAsync(w.ids.p, ids_host, (size_t)m * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        ids_dev = w.ids.as<int64_t>();
    }
    const void* P;
    const float* Pn;
    B2_TRY(point_set(idx, ids_dev, m, w, P, Pn, st));
    // training set (faiss ClusteringParameters: max_points_per_centroid = 256)
    int64_t nx = m;
    const void* T = P;
    const float* Tn = Pn;
    const int64_t max_pts = (int64_t)k * 256;
    std::vector<int64_t> perm;
    if (!full_lloyd && nx > max_pts) {
        rand_perm_prefix(perm, nx, max_pts, seed);
        nx = max_pts;
        B2_TRY(w.perm.ensure((size_t)nx * sizeof(int64_t)));
        B2_TRY(w.train.ensure((size_t)nx * d * es));
        B2_TRY(w.train_norm2.ensure((size_t)nx * sizeof(float)));
        B2_TRY(w.scalar.ensure(64));
        B2_CUDA(cudaMemcpyAsync(w.perm.p, perm.data(), (size_t)nx * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        int* err = reinterpret_cast<int*>(w.scalar.as<char>() + 16);
        B2_TRY(launch_gather_rows(P, idx->dtype, d, w.perm.as<int64_t>(), nx, m, w.train.p, err, st));
        B2_TRY(launch_row_norms(w.train.p, idx->dtype, nx, d, w.train_norm2.as<float>(), w.scalar.as<float>() + 8, st));
        B2_CUDA(cudaStreamSynchronize(st));  // `perm` (host vector) is reused below
        T = w.train.p;
        Tn = w.train_norm2.as<float>();
    }
    B2_TRY(w.cent[0].ensure((size_t)k * d * sizeof(float)));
    B2_TRY(w.cent[1].ensure((size_t)k * d * sizeof(float)));
    int cur = 0;
    if (nx == k) {
        // "Number of training points same as number of centroids, just copying"
        rows_to_f32_kernel<<<148, 256, 0, st>>>(T, idx->dtype, d, nullptr, k, w.cent[0].as<float>());
        B2_LAUNCH_CHECK();
    } else {
        rand_perm_prefix(perm, nx, k, seed + 1);
        B2_TRY(w.perm.ensure((size_t)k * sizeof(int64_t)));
        B2_CUDA(cudaMemcpyAsync(w.perm.p, perm.data(), (size_t)k * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        rows_to_f32_kernel<<<148, 256, 0, st>>>(T, idx->dtype, d, w.perm.as<int64_t>(), k, w.cent[0].as<float>());
        B2_LAUNCH_CHECK();
        B2_CUDA(cudaStreamSynchronize(st));
        B2_TRY(w.assign.ensure((size_t)nx * sizeof(int64_t)));
        B2_TRY(w.obj.ensure((size_t)std::max(niter, 1) * sizeof(double)));
        B2_CUDA(cudaMemsetAsync(w.obj.p, 0, (size_t)std::max(niter, 1) * sizeof(double), st));
        tm.lap(0);
        for (int it = 0; it < niter; ++it) {
            int64_t n2 = 0;
            B2_TRY(assign_points(idx, T, Tn, nx, w.cent[cur].as<float>(), k, w, w.assign.as<int64_t>(), st, &n2));
            tm.lap(1);
            tm.second_level += n2;
            if (tm.on && idx->last_filter_ms > 0) tm.acc[2] += idx->last_filter_ms;
            B2_TRY(update_centroids(idx, T, nullptr, nx, w.assign.as<int64_t>(), k, w, out_obj ? w.cent[cur].as<float>() : nullptr,
                                    w.cent[cur ^ 1].as<float>(), w.obj.as<double>() + it, st, /*normalize=*/1));
            km_split_kernel<<<1, 256, 0, st>>>(d, k, nx, w.hassign.as<float>(), w.cent[cur ^ 1].as<float>());
            B2_LAUNCH_CHECK();
            cur ^= 1;
            tm.lap(3);
        }
    }
    tm.lap(0);
    // lotus/utils.py:65 kmeans.index.search(vec_set, 1) over ALL m points
    B2_TRY(w.fin_assign.ensure((size_t)std::max<int64_t>(m, 1) * sizeof(int64_t)));
    B2_TRY(assign_points(idx, P, Pn, m, w.cent[cur].as<float>(), k, w, w.fin_assign.as<int64_t>(), st));
    B2_CUDA(cudaMemcpyAsync(out_assign, w.fin_assign.p, (size_t)m * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    if (out_centroids) B2_CUDA(cudaMemcpyAsync(out_centroids, w.cent[cur].p, (size_t)k * d * sizeof(float), cudaMemcpyDeviceToHost, st));
    std::vector<double> h_obj(std::max(niter, 1), 0.0);
    if (out_obj && nx != k && niter > 0) B2_CUDA(cudaMemcpyAsync(h_obj.data(), w.obj.p, (size_t)niter * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (cudaStreamSynchronize(st) != cudaSuccess) {
        set_error("k-means failed on the device: %s", cudaGetErrorString(cudaGetLastError()));
        return B2_ECUDA;
    }
    tm.lap(5);
    tm.report(m, nx, k, d, niter);
    if (out_obj)
        for (int it = 0; it < niter; ++it) out_obj[it] = (float)h_obj[it];
    return B2_OK;
}

KmWork& work_of(b2_index* idx) {
    if (!idx->km) idx->km = new KmWork();
    return *idx->km;
}

int check_ids_host(b2_index* idx, const int64_t* ids, int64_t m) {
    if (!ids) return B2_OK;
    for (int64_t i = 0; i < m; ++i)
        if (ids[i] < 0 || ids[i] >= idx->n) {
            set_error("ids contains a position outside [0, %lld)", (long long)idx->n);
            return B2_ERANGE;
        }
    return B2_OK;
}

}  // namespace
}  // namespace b2

using namespace b2;

extern "C" {

int b2_kmeans(b2_index* idx, const int64_t* ids, int64_t m, int32_t k, int32_t niter, int64_t seed, int32_t full_lloyd,
              int64_t* out_assign, float* out_centroids, float* out_obj) {
    if (!idx) { set_error("Index not loaded"); return B2_EINVAL; }
    if (!ids) m = idx->n;
    if (k <= 0 || niter < 0 || m < 0 || !out_assign) { set_error("bad k-means arguments (k=%d niter=%d m=%lld)", k, niter, (long long)m); return B2_EINVAL; }
    if (m < k) { set_error("Number of training points (%lld) should be at least as large as number of clusters (%d)", (long long)m, k); return B2_EINVAL; }
    if (k > 0x7fffff00 / 2) { set_error("k=%d too large", k); return B2_ERANGE; }
    B2_TRY(check_ids_host(idx, ids, m));
    DeviceGuard guard(idx->device);
    KmWork& w = work_of(idx);
    const int rc = kmeans_impl(idx, ids, m, k, niter, seed, full_lloyd, out_assign, out_centroids, out_obj, w);
    cudaStreamSynchronize(idx->stream);
    // the large per-call buffers go back; the small ones stay with the handle for the next call
    DevBuf* big[] = {&w.pts, &w.pts_norm2, &w.train, &w.train_norm2, &w.assign, &w.members, &w.flag_ids, &w.hard_ids, &w.sub, &w.fin_assign, &w.ids, &w.perm};
    for (DevBuf* b : big) b->release();
    return rc;
}

int b2_kmeans_assign_dev(b2_index* idx, const int64_t* ids_dev, int64_t m, const float* centroids_dev, int32_t k, int64_t* assign_dev,
                         float* dist_dev, void* stream) {
    if (!idx) { set_error("Index not loaded"); return B2_EINVAL; }
    if (!ids_dev) m = idx->n;
    if (k <= 0 || m < 0 || !centroids_dev || (m > 0 && !assign_dev)) { set_error("bad arguments"); return B2_EINVAL; }
    if (m == 0) return B2_OK;
    DeviceGuard guard(idx->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    KmWork& w = work_of(idx);
    const void* P;
    const float* Pn;
    B2_TRY(point_set(idx, ids_dev, m, w, P, Pn, st));
    B2_TRY(assign_points(idx, P, Pn, m, centroids_dev, k, w, assign_dev, st));
    if (dist_dev) B2_TRY(launch_exact_l2_assigned(P, idx->dtype, m, idx->d, centroids_dev, assign_dev, dist_dev, st));
    B2_CUDA(cudaStreamSynchronize(st));
    return B2_OK;
}

int b2_kmeans_accumulate_dev(b2_index* idx, const int64_t* ids_dev, int64_t m, const int64_t* assign_dev, int32_t k,
                             const float* centroids_dev, float* sums_dev, float* counts_dev, double* obj_dev, void* stream) {
    if (!idx) { set_error("Index not loaded"); return B2_EINVAL; }
    if (!ids_dev) m = idx->n;
    if (k <= 0 || m < 0 || (m > 0 && !assign_dev) || !sums_dev || !counts_dev) { set_error("bad arguments"); return B2_EINVAL; }
    if (obj_dev && !centroids_dev) { set_error("the objective needs the centroids the assignment was made against"); return B2_EINVAL; }
    DeviceGuard guard(idx->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    KmWork& w = work_of(idx);
    B2_TRY(update_centroids(idx, idx->store.p, ids_dev, m, assign_dev, k, w, obj_dev ? centroids_dev : nullptr, sums_dev, obj_dev, st,
                            /*normalize=*/0));
    B2_CUDA(cudaMemcpyAsync(counts_dev, w.hassign.p, (size_t)k * sizeof(float), cudaMemcpyDeviceToDevice, st));
    B2_CUDA(cudaStreamSynchronize(st));
    return B2_OK;
}

int b2_kmeans_accumulate(b2_index* idx, const int64_t* ids, int64_t m, const int64_t* assign, int32_t k, float* out_sums,
                         float* out_counts) {
    if (!idx) { set_error("Index not loaded"); return B2_EINVAL; }
    if (!ids) m = idx->n;
    if (k <= 0 || m < 0 || !assign || !out_sums || !out_counts) { set_error("bad arguments"); return B2_EINVAL; }
    for (int64_t i = 0; i < m; ++i)
        if (assign[i] < 0 || assign[i] >= k) { set_error("assign[%lld] = %lld outside [0, %d)", (long long)i, (long long)assign[i], k); return B2_ERANGE; }
    B2_TRY(check_ids_host(idx, ids, m));
    DeviceGuard guard(idx->device);
    cudaStream_t st = idx->stream;
    KmWork& w = work_of(idx);
    DevBuf d_assign, d_sums, d_counts;
    int rc = d_assign.ensure((size_t)std::max<int64_t>(m, 1) * sizeof(int64_t));
    if (rc == B2_OK) rc = d_sums.ensure((size_t)k * idx->d * sizeof(float));
    if (rc == B2_OK) rc = d_counts.ensure((size_t)k * sizeof(float));
    const int64_t* ids_dev = nullptr;
    if (rc == B2_OK && ids) {
        rc = w.ids.ensure((size_t)std::max<int64_t>(m, 1) * sizeof(int64_t));
        if (rc == B2_OK) {
            cudaMemcpyAsync(w.ids.p, ids, (size_t)m * sizeof(int64_t), cudaMemcpyHostToDevice, st);
            ids_dev = w.ids.as<int64_t>();
        }
    }
    if (rc == B2_OK) {
        cudaMemcpyAsync(d_assign.p, assign, (size_t)m * sizeof(int64_t), cudaMemcpyHostToDevice, st);
        rc = b2_kmeans_accumulate_dev(idx, ids_dev, m, d_assign.as<int64_t>(), k, nullptr, d_sums.as<float>(), d_counts.as<float>(), nullptr, st);
    }
    if (rc == B2_OK) {
        cudaMemcpyAsync(out_sums, d_sums.p, (size_t)k * idx->d * sizeof(float), cudaMemcpyDeviceToHost, st);
        cudaMemcpyAsync(out_counts, d_counts.p, (size_t)k * sizeof(float), cudaMemcpyDeviceToHost, st);
        if (cudaStreamSynchronize(st) != cudaSuccess) {
            set_error("k-means accumulate failed on the device: %s", cudaGetErrorString(cudaGetLastError()));
            rc = B2_ECUDA;
        }
    } else {
        cudaStreamSynchronize(st);
    }
    d_assign.release();
    d_sums.release();
    d_counts.release();
    return rc;
}

int b2_kmeans_assign(b2_index* idx, const int64_t* ids, int64_t m, const float* centroids, int32_t k, int64_t* out_assign,
                     float* out_dist) {
    if (!idx) { set_error("Index not loaded"); return B2_EINVAL; }
    if (!ids) m = idx->n;
    if (k <= 0 || m < 0 || !centroids || (m > 0 && !out_assign)) { set_error("bad arguments"); return B2_EINVAL; }
    if (m == 0) return B2_OK;
    B2_TRY(check_ids_host(idx, ids, m));
    DeviceGuard guard(idx->device);
    cudaStream_t st = idx->stream;
    const int d = idx->d;
    KmWork& w = work_of(idx);
    DevBuf cent, dis, asg;
    auto cleanup = [&]() { cudaStreamSynchronize(st); cent.release(); dis.release(); asg.release(); w.pts.release(); w.pts_norm2.release(); };
    int rc = cent.ensure((size_t)k * d * sizeof(float));
    if (rc == B2_OK && out_dist) rc = dis.ensure((size_t)m * sizeof(float));
    if (rc == B2_OK) rc = asg.ensure((size_t)m * sizeof(int64_t));
    const int64_t* ids_dev = nullptr;
    if (rc == B2_OK && ids) {
        rc = w.ids.ensure((size_t)m * sizeof(int64_t));
        if (rc == B2_OK) {
            cudaMemcpyAsync(w.ids.p, ids, (size_t)m * sizeof(int64_t), cudaMemcpyHostToDevice, st);
            ids_dev = w.ids.as<int64_t>();
        }
    }
    if (rc == B2_OK) {
        cudaMemcpyAsync(cent.p, centroids, (size_t)k * d * sizeof(float), cudaMemcpyHostToDevice, st);
        rc = b2_kmeans_assign_dev(idx, ids_dev, m, cent.as<float>(), k, asg.as<int64_t>(), out_dist ? dis.as<float>() : nullptr, st);
    }
    if (rc == B2_OK) {
        cudaMemcpyAsync(out_assign, asg.p, (size_t)m * sizeof(int64_t), cudaMemcpyDeviceToHost, st);
        if (out_dist) cudaMemcpyAsync(out_dist, dis.p, (size_t)m * sizeof(float), cudaMemcpyDeviceToHost, st);
        if (cudaStreamSynchronize(st) != cudaSuccess) {
            set_error("k-means assignment failed on the device: %s", cudaGetErrorString(cudaGetLastError()));
            rc = B2_ECUDA;
        }
    }
    cleanup();
    return rc;
}

}  // extern "C"
