// knn_exact.cu — the exact side of the search pipeline (everything that decides the reported result).
//
//   finalize_kernel   : per query (one warp): merge the per-split candidate lists of the tcgen05 filter with a
//                       warp-shuffle bitonic network, re-score the KP survivors in the canonical fp64 order,
//                       sort them, apply faiss's heap tie rule, and CERTIFY the result against everything the
//                       filter discarded (rigorous error margin). Uncertified queries are flagged.
//   dense_topk        : exact brute force for flagged queries and for k beyond the filter's capacity:
//                       canonical scores for a batch of queries, block radix select, ordered tie collection.
//   merge_topk_kernel : single-kernel k-way merge of per-shard (score, idx) lists after the NCCL all-gather.
//   plus query preparation, row norms, padding/conversion and row gather (faiss_vs.py:38-41).
//
// Canonical score (bit-for-bit what oracle/faiss_flat.c `orc_dot_canonical` / `orc_l2_canonical` compute):
// element i is accumulated by lane (i>>2)&31 in increasing i with fp64 fma; the 32 partials are combined by
// a 16,8,4,2,1 xor-butterfly; the double is rounded once to fp32.
#include <cub/cub.cuh>

#include "canonical.cuh"
#include "common.cuh"

namespace b2 {

namespace {

constexpr uint64_t KEY_WORST = ~0ull;

struct MergeOffsets {  // global id of row 0 of every shard (by value: at most one box of GPUs)
    static constexpr int MAX = 16;
    int64_t v[MAX];
};

// ---- warp-shuffle bitonic sort of 32*R u64 keys, element e = r*32 + lane, ascending ------------------------
template <int R>
__device__ __forceinline__ void warp_bitonic_sort(uint64_t (&key)[R], int lane) {
#pragma unroll
    for (int k = 2; k <= 32 * R; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32) {
                const int jr = j >> 5;
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int rp = r ^ jr;
                    if (rp > r) {
                        const bool up = (((r * 32) & k) == 0);  // k >= 64 here: independent of lane
                        const uint64_t a = key[r], b = key[rp];
                        const bool sw = (a > b) == up;
                        key[r] = sw ? b : a;
                        key[rp] = sw ? a : b;
                    }
                }
            } else {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int e = r * 32 + lane;
                    const bool up = ((e & k) == 0);
                    const uint64_t other = __shfl_xor_sync(FULL, key[r], j);
                    const bool lower = ((lane & j) == 0);
                    const bool keep_min = (lower == up);
                    const uint64_t mn = key[r] < other ? key[r] : other;
                    const uint64_t mx = key[r] < other ? other : key[r];
                    key[r] = keep_min ? mn : mx;
                }
            }
        }
    }
}

// Sorts a BITONIC sequence of 32*R keys ascending (the merge half of the network: log2(32R) stages instead of the
// full sort's log^2).
template <int R>
__device__ __forceinline__ void warp_bitonic_merge(uint64_t (&key)[R], int lane) {
#pragma unroll
    for (int j = 16 * R; j > 0; j >>= 1) {
        if (j >= 32) {
            const int jr = j >> 5;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int rp = r ^ jr;
                if (rp > r) {
                    const uint64_t a = key[r], b = key[rp];
                    key[r] = a < b ? a : b;
                    key[rp] = a < b ? b : a;
                }
            }
        } else {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const uint64_t other = __shfl_xor_sync(FULL, key[r], j);
                const bool lower = ((lane & j) == 0);
                const uint64_t mn = key[r] < other ? key[r] : other;
                const uint64_t mx = key[r] < other ? other : key[r];
                key[r] = lower ? mn : mx;
            }
        }
    }
}

// buf (sorted ascending, 32*R keys) <- the 32*R smallest of buf U chunk (chunk sorted ascending), sorted again.
// Returns the smallest key that was dropped (KEY_WORST if none): min(buf[e], chunk[N-1-e]) keeps exactly the lower half
// of the union and is bitonic, so one merge pass re-sorts it.
template <int R>
__device__ __forceinline__ uint64_t warp_merge_keep_low(uint64_t (&buf)[R], const uint64_t (&chunk)[R], int lane) {
    uint64_t best_drop = KEY_WORST;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint64_t rev = __shfl_sync(FULL, chunk[R - 1 - r], 31 - lane);  // chunk[N-1-e] for e = r*32 + lane
        const uint64_t a = buf[r];
        const uint64_t hi = a < rev ? rev : a;
        buf[r] = a < rev ? a : rev;
        best_drop = hi < best_drop ? hi : best_drop;
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const uint64_t o = __shfl_xor_sync(FULL, best_drop, off);
        best_drop = o < best_drop ? o : best_drop;
    }
    warp_bitonic_merge<R>(buf, lane);
    return best_drop;
}

// ---- small utility kernels -------------------------------------------------------------------------------------
// one element of a filter operand in out_dtype (round to nearest even); false when the result is not finite
__device__ __forceinline__ bool store_operand(void* out, int out_dtype, int64_t t, float v) {
    if (out_dtype == B2_F32) {
        reinterpret_cast<float*>(out)[t] = v;
        return true;
    }
    if (out_dtype == B2_F16) {
        __half h = __float2half_rn(v);
        const bool fin = !__hisinf(h) && !__hisnan(h);
        reinterpret_cast<__half*>(out)[t] = fin ? h : __float2half_rn(0.f);
        return fin;
    }
    reinterpret_cast<__nv_bfloat16*>(out)[t] = __float2bfloat16_rn(v);
    return true;
}

__global__ void prep_queries_kernel(const void* q, int q_dtype, int64_t nq, int d, void* out, int out_dtype, int64_t pitch,
                                    int32_t* bad) {
    const int64_t total = nq * pitch;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = t / pitch;
        const int c = (int)(t - r * pitch);
        const float v = c < d ? elem_f32(q, q_dtype, (size_t)(r * d + c)) : 0.f;
        if (!store_operand(out, out_dtype, t, v) && bad) bad[r] = 1;
    }
}

__global__ void row_norms_kernel(const void* x, int dtype, int64_t n, int d, float* norm2, float* max_norm) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const bool vec = (d % 4) == 0;
    const size_t esz = dtype == B2_F32 ? 4 : 2;
    float local_max = 0.f;
    for (int64_t j = warp; j < n; j += nwarps) {
        const char* row = reinterpret_cast<const char*>(x) + (size_t)j * d * esz;
        double acc = 0.0;
        const int ngroups = (d + 3) >> 2;
        for (int g = lane; g < ngroups; g += 32) {
            float v[4];
            load_group(row, dtype, g, d, vec, v);
#pragma unroll
            for (int e = 0; e < 4; ++e) acc = fma((double)v[e], (double)v[e], acc);
        }
        const double tot = butterfly_sum(acc);
        if (lane == 0) norm2[j] = (float)tot;
        local_max = fmaxf(local_max, (float)sqrt(tot) * (1.0f + 1e-6f));
    }
    if (lane == 0 && local_max > 0.f) atomicMax(reinterpret_cast<int*>(max_norm), __float_as_int(local_max));
}

__global__ void convert_pad_kernel(const void* x, int dtype, int64_t n, int d, void* out, int out_dtype, int64_t pitch, int32_t* bad) {
    const int64_t total = n * pitch;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = t / pitch;
        const int c = (int)(t - r * pitch);
        const float v = c < d ? elem_f32(x, dtype, (size_t)(r * d + c)) : 0.f;
        if (!store_operand(out, out_dtype, t, v) && bad) *bad = 1;
    }
}

// out[i,:] = x[ids[i],:] — one warp per row, 16-byte copies when the row size allows
__global__ void gather_rows_kernel(const char* x, size_t row_bytes, const int64_t* ids, int64_t m, int64_t n, char* out,
                                   int* err_flag) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp; i < m; i += nwarps) {
        const int64_t id = ids[i];
        if (id < 0 || id >= n) {
            if (lane == 0) atomicExch(err_flag, 1);
            continue;
        }
        const char* src = x + (size_t)id * row_bytes;
        char* dst = out + (size_t)i * row_bytes;
        if ((row_bytes & 15) == 0) {
            const int4* s4 = reinterpret_cast<const int4*>(src);
            int4* d4 = reinterpret_cast<int4*>(dst);
            for (size_t t = lane; t < row_bytes / 16; t += 32) d4[t] = __ldg(s4 + t);
        } else {
            const uint16_t* s2 = reinterpret_cast<const uint16_t*>(src);
            uint16_t* d2 = reinterpret_cast<uint16_t*>(dst);
            for (size_t t = lane; t < row_bytes / 2; t += 32) d2[t] = s2[t];
        }
    }
}

// Canonical partials of U rows at once (vectorisable rows only): the U independent row loads of a step are issued
// back to back, so each lane keeps U gathers in flight. Per row the accumulation order is exactly canonical_partial's.
template <bool IS_L2, int DT, int U>  // DT: element type of the rows (B2_F32, B2_BF16 or B2_F16)
__device__ __forceinline__ void canonical_partial_multi(const float* q_s, const char* const (&rows)[U], int d, int lane,
                                                        double (&acc)[U]) {
#pragma unroll
    for (int u = 0; u < U; ++u) acc[u] = 0.0;
    const int ngroups = d >> 2;
    for (int g = lane; g < ngroups; g += 32) {
        float x[U][4];
        if constexpr (DT == B2_F16) {
            uint2 t[U];
#pragma unroll
            for (int u = 0; u < U; ++u) t[u] = __ldg(reinterpret_cast<const uint2*>(rows[u]) + g);
#pragma unroll
            for (int u = 0; u < U; ++u) f16x4_to_f32(t[u], x[u]);
        } else if constexpr (DT == B2_BF16) {
            uint2 t[U];
#pragma unroll
            for (int u = 0; u < U; ++u) t[u] = __ldg(reinterpret_cast<const uint2*>(rows[u]) + g);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                x[u][0] = __uint_as_float(t[u].x << 16);
                x[u][1] = __uint_as_float(t[u].x & 0xffff0000u);
                x[u][2] = __uint_as_float(t[u].y << 16);
                x[u][3] = __uint_as_float(t[u].y & 0xffff0000u);
            }
        } else {
            float4 t[U];
#pragma unroll
            for (int u = 0; u < U; ++u) t[u] = __ldg(reinterpret_cast<const float4*>(rows[u]) + g);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                x[u][0] = t[u].x; x[u][1] = t[u].y; x[u][2] = t[u].z; x[u][3] = t[u].w;
            }
        }
        const float4 q4 = *reinterpret_cast<const float4*>(q_s + 4 * g);
        const float qq[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
        for (int u = 0; u < U; ++u) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                if (IS_L2) {
                    const double diff = (double)qq[e] - (double)x[u][e];
                    acc[u] = fma(diff, diff, acc[u]);
                } else {
                    acc[u] = fma((double)qq[e], (double)x[u][e], acc[u]);
                }
            }
        }
    }
}

// ---- finalize ------------------------------------------------------------------------------------------------
struct FinalizeParams {
    const void* store;
    const void* q;
    const float* cand_score;
    const int32_t* cand_id;
    const float* cand_thr;
    const int64_t* id_map;
    float* out_scores;
    int64_t* out_idx;
    int32_t* flags;
    int32_t* sel;        // [nq] queries whose certificate failed, in arbitrary order (nullable)
    int32_t* sel_count;  // number of entries in sel (device counter, zeroed by the caller)
    int64_t nq;
    int64_t id_offset;
    int32_t d, dtype, q_dtype, metric, k, kp, n_splits;  // n_splits = number of candidate lists per query, kp = survivors kept
    int32_t list_len;                                    // entries per candidate list (<= 32*R)
    float rel_eps, abs_eps, max_norm;  // filter error: filter_ip_err(rel_eps, abs_eps, ||q||, ||x||)
    const float* max_norm_dev;  // nullable: overrides max_norm
    const int32_t* q_bad;       // nullable: queries whose filter operand is not finite (prep_queries): never certified
    const float* hint;          // nullable: per query, a lower bound (filter-score space) on the k-th exact score of the WHOLE
                                // row-sharded search (b2_index_search_stage1_dev + all-reduce MIN over the ranks)
};

constexpr int FIN_WARPS = 4;

template <int R>  // 32*R >= KP candidates survive the merge
__global__ void __launch_bounds__(FIN_WARPS * 32) finalize_kernel(const FinalizeParams p) {
    constexpr int NC = 32 * R;
    extern __shared__ __align__(16) uint8_t fsm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int d4 = ((p.d + 3) >> 2) << 2;
    const size_t per_warp = (size_t)d4 * 4 + (size_t)NC * (4 + 4 + 8);
    uint8_t* base = fsm + warp * per_warp;
    uint64_t* s_keys = reinterpret_cast<uint64_t*>(base);         // [NC] sorted exact keys
    float* q_s = reinterpret_cast<float*>(base + (size_t)NC * 8);  // [d4]
    int32_t* s_id = reinterpret_cast<int32_t*>(q_s + d4);         // [NC]
    float* s_ex = reinterpret_cast<float*>(s_id + NC);            // [NC]

    const int64_t q = blockIdx.x * (int64_t)FIN_WARPS + warp;
    if (q >= p.nq) return;
    const float max_norm = p.max_norm_dev ? __ldg(p.max_norm_dev) : p.max_norm;
    const bool is_l2 = p.metric == B2_METRIC_L2;
    const bool vec = (p.d % 4) == 0;
    const size_t esz = p.dtype == B2_F32 ? 4 : 2;

    // 1. query -> smem (fp32, exact upcast for bf16) and its canonical squared norm
    for (int i = lane; i < d4; i += 32) q_s[i] = i < p.d ? elem_f32(p.q, p.q_dtype, (size_t)q * p.d + i) : 0.f;
    __syncwarp();
    double qacc = 0.0;
    for (int g = lane; g < (d4 >> 2); g += 32) {
#pragma unroll
        for (int e = 0; e < 4; ++e) qacc = fma((double)q_s[4 * g + e], (double)q_s[4 * g + e], qacc);
    }
    const double qn2 = butterfly_sum(qacc);

    // 2. merge the candidate lists by filter score (larger is better for both metrics): chunks of 32*R keys (as many
    //    whole lists as fit) are sorted with the bitonic network and folded into the running best 32*R with one
    //    compare-with-reversed + bitonic-merge pass each (instead of re-sorting 2*32*R keys per list)
    uint64_t keys[R];
    float bound = -INFINITY;
    {
        const int lists_per_chunk = max(1, NC / p.list_len);
        const size_t qbase = (size_t)q * p.n_splits;
        bool first = true;
        for (int s0 = 0; s0 < p.n_splits; s0 += lists_per_chunk) {
            uint64_t chunk[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int e = r * 32 + lane;
                const int li = e / p.list_len, pos = e - li * p.list_len;
                uint64_t kk = KEY_WORST;
                if (li < lists_per_chunk && s0 + li < p.n_splits) {
                    const size_t off = (qbase + s0 + li) * p.list_len + pos;
                    const int32_t id = p.cand_id[off];
                    if (id >= 0) kk = ((uint64_t)(~f32_ord(p.cand_score[off])) << 32) | (uint32_t)id;
                }
                chunk[r] = kk;
            }
            for (int li = lane; li < lists_per_chunk && s0 + li < p.n_splits; li += 32) bound = fmaxf(bound, p.cand_thr[qbase + s0 + li]);
            {  // lists of a query unit that swept the corpus as ONE item are empty beyond split 0: nothing to sort or fold
                bool any_key = false;
#pragma unroll
                for (int r = 0; r < R; ++r) any_key |= chunk[r] != KEY_WORST;
                if (!__any_sync(FULL, any_key) && !first) continue;
            }
            warp_bitonic_sort<R>(chunk, lane);
            if (first) {
#pragma unroll
                for (int r = 0; r < R; ++r) keys[r] = chunk[r];
                first = false;
            } else {
                // best discarded candidate bounds everything dropped by this fold
                const uint64_t drop = warp_merge_keep_low<R>(keys, chunk, lane);
                if (drop != KEY_WORST) bound = fmaxf(bound, f32_unord(~(uint32_t)(drop >> 32)));
            }
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) bound = fmaxf(bound, __shfl_xor_sync(FULL, bound, off));
    }
    // margin between a filter score and the exact score it stands for (same quantity the certificate uses below)
    const double qn_m = sqrt(qn2), mx_m = (double)max_norm;
    const double ip_err = filter_ip_err((double)p.rel_eps, (double)p.abs_eps, qn_m, mx_m);
    const double eps_f = is_l2 ? 2.0 * ip_err + 2.4e-7 * (mx_m * mx_m + 2.0 * qn_m * mx_m) + 1e-30 : ip_err + 1e-30;
    // Pruning before the (expensive) re-score: the k best survivors BY FILTER SCORE have exact scores >= t_k - eps, so a
    // survivor whose filter score is below t_k - 2 eps is strictly worse than k others: it cannot enter or tie the top k.
#pragma unroll
    for (int r = 0; r < R; ++r) s_ex[r * 32 + lane] = keys[r] == KEY_WORST ? -INFINITY : f32_unord(~(uint32_t)(keys[r] >> 32));
    __syncwarp();
    float cut = -INFINITY;
    if (p.k <= NC) {
        const float tk = s_ex[p.k - 1];
        if (tk > -INFINITY) cut = (float)((double)tk - 2.0 * eps_f - 4.8e-7 * fabs((double)tk));
    }
    // Row-sharded search: k rows with exact score >= hint exist somewhere in the index, so a local row whose exact score is surely
    // below that (filter + eps < hint) cannot enter or tie the merged top k: do not re-score it (this is what lets 8 ranks
    // re-score ~k/8 rows each instead of k+2).
    const double hint = p.hint ? (double)p.hint[q] : -INFINITY;
    const double hint_slack = 4.8e-7 * fabs(hint) + (is_l2 ? 4.8e-7 * qn2 : 0.0);
    if (hint > -INFINITY) cut = fmaxf(cut, (float)(hint - eps_f - hint_slack));
    __syncwarp();
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int e = r * 32 + lane;
        const bool keep = keys[r] != KEY_WORST && f32_unord(~(uint32_t)(keys[r] >> 32)) >= cut;
        s_id[e] = keep ? (int32_t)(uint32_t)(keys[r] & 0xffffffffu) : -1;
    }
    __syncwarp();

    // 3. canonical re-scoring of the surviving candidates, four rows per step (survivors are sorted by filter score,
    //    so the pruned tail of the list is skipped as soon as a whole step is empty)
    for (int c0 = 0; c0 < NC; c0 += 4) {
        double part[4];
        int32_t ids[4];
        bool any_valid = false;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            ids[u] = s_id[c0 + u];
            any_valid |= ids[u] >= 0;
        }
        if (!any_valid) break;
        if (vec) {
            // interleaved gather of the four rows (an invalid slot re-reads the first row of the step: a cache hit)
            const char* rows[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                rows[u] = reinterpret_cast<const char*>(p.store) + (size_t)(ids[u] >= 0 ? ids[u] : ids[0]) * p.d * esz;
            if (p.dtype == B2_BF16) {
                if (is_l2) canonical_partial_multi<true, B2_BF16, 4>(q_s, rows, p.d, lane, part);
                else canonical_partial_multi<false, B2_BF16, 4>(q_s, rows, p.d, lane, part);
            } else if (p.dtype == B2_F16) {
                if (is_l2) canonical_partial_multi<true, B2_F16, 4>(q_s, rows, p.d, lane, part);
                else canonical_partial_multi<false, B2_F16, 4>(q_s, rows, p.d, lane, part);
            } else {
                if (is_l2) canonical_partial_multi<true, B2_F32, 4>(q_s, rows, p.d, lane, part);
                else canonical_partial_multi<false, B2_F32, 4>(q_s, rows, p.d, lane, part);
            }
        } else {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                part[u] = 0.0;
                if (ids[u] >= 0) {
                    const char* row = reinterpret_cast<const char*>(p.store) + (size_t)ids[u] * p.d * esz;
                    part[u] = is_l2 ? canonical_partial<true>(q_s, row, p.dtype, p.d, vec, lane)
                                    : canonical_partial<false>(q_s, row, p.dtype, p.d, vec, lane);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const double tot = butterfly_sum(part[u]);
            if (lane == 0) s_ex[c0 + u] = (float)tot;
        }
    }
    __syncwarp();

    // 4. exact keys: (score best first, then faiss's tie order: id ascending for L2, id descending for IP)
    uint64_t ek[R];
    int nvalid = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int e = r * 32 + lane;
        const int32_t id = s_id[e];
        if (id >= 0) {
            const uint32_t tie = is_l2 ? (uint32_t)id : ~(uint32_t)id;
            ek[r] = ((uint64_t)best_first_key(s_ex[e], p.metric) << 32) | tie;
            nvalid++;
        } else {
            ek[r] = KEY_WORST;
        }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) nvalid += __shfl_xor_sync(FULL, nvalid, off);
    warp_bitonic_sort<R>(ek, lane);
#pragma unroll
    for (int r = 0; r < R; ++r) s_keys[r * 32 + lane] = ek[r];
    __syncwarp();

    // 5. faiss heap rule at rank k (DESIGN.md §Ties) -> output positions
    const int k = p.k;
    const int nout = nvalid < k ? nvalid : k;
    int c = nout, m = 0, t = 0, r_keep = 0;  // better-than-v count, ties at v, ties inside the first-k-by-id window
    uint32_t vkey = 0;
    if (nvalid > k) {
        vkey = (uint32_t)(s_keys[k - 1] >> 32);
        int cc = 0, mm = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const uint32_t hk = (uint32_t)(ek[r] >> 32);
            const bool valid = ek[r] != KEY_WORST;
            cc += (valid && hk < vkey) ? 1 : 0;
            mm += (valid && hk == vkey) ? 1 : 0;
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            cc += __shfl_xor_sync(FULL, cc, off);
            mm += __shfl_xor_sync(FULL, mm, off);
        }
        c = cc;
        m = mm;
        r_keep = k - c;
        t = m;
        if (!is_l2 && m > r_keep) {
            // ties inside the first k (by ascending id) elements of S = {score >= v}
            int tt = 0;
            for (int e = c + lane; e < c + m; e += 32) {
                const uint32_t id_e = ~(uint32_t)(s_keys[e] & 0xffffffffu);
                int rank = 1;
                for (int f = 0; f < c + m; ++f) rank += (~(uint32_t)(s_keys[f] & 0xffffffffu) < id_e) ? 1 : 0;
                tt += rank <= k ? 1 : 0;
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) tt += __shfl_xor_sync(FULL, tt, off);
            t = tt;
        }
    }
    // sorted ties sit at [c, c+m): L2 ascending id -> keep the first r; IP descending id (e_m .. e_1) -> keep e_t .. e_{t-r+1}
    const int tie_src0 = (is_l2 || nvalid <= k) ? c : c + m - t;

    // 6. certification against everything the filter discarded
    // a query the filter could not see as finite operands has meaningless filter scores: the exact path answers it
    bool certified = !(p.q_bad && p.q_bad[q]);
    // everything the filter discarded scores (exactly) at most bound + eps: below the sharded search's k-th score -> irrelevant
    const bool hint_ok = hint > -INFINITY && ((double)bound + eps_f) < hint - hint_slack;
    if (certified && bound > -INFINITY && !hint_ok) {
        if (nvalid < k) {
            certified = false;  // cannot happen (lists only overflow when full); be safe
        } else {
            const double qn = sqrt(qn2);
            const double v = (double)best_first_unkey((uint32_t)(s_keys[k - 1] >> 32), p.metric);
            if (!is_l2) {
                const double eps = filter_ip_err((double)p.rel_eps, (double)p.abs_eps, qn, (double)max_norm) + 1e-30;
                certified = ((double)bound + eps) < v;
            } else {
                const double mx = (double)max_norm;
                const double eps_s = 2.0 * filter_ip_err((double)p.rel_eps, (double)p.abs_eps, qn, mx) + 2.4e-7 * (mx * mx + 2.0 * qn * mx) + 1e-30;
                // discarded rows have exact L2 >= qn2 - (bound + eps_s); allow for the fp32 rounding of v
                certified = (qn2 - (double)bound - eps_s) > v * (1.0 + 2.4e-7) + 1e-30;
            }
        }
    }

    // 7. write
    const float pad = is_l2 ? FLT_MAX : -FLT_MAX;
    for (int o = lane; o < k; o += 32) {
        float sc = pad;
        int64_t oid = -1;
        if (o < nout) {
            const int src = o < c ? o : tie_src0 + (o - c);
            const uint64_t kk = s_keys[src];
            const uint32_t lo = (uint32_t)(kk & 0xffffffffu);
            const int32_t id = (int32_t)(is_l2 ? lo : ~lo);
            sc = best_first_unkey((uint32_t)(kk >> 32), p.metric);
            oid = p.id_map ? p.id_map[id] : (int64_t)id + p.id_offset;
        }
        p.out_scores[(size_t)q * k + o] = sc;
        p.out_idx[(size_t)q * k + o] = oid;
    }
    if (lane == 0) {
        p.flags[q] = certified ? 0 : 1;
        if (!certified && p.sel) p.sel[atomicAdd(p.sel_count, 1)] = (int32_t)q;
    }
}

// ---- dense exact path -----------------------------------------------------------------------------------------
// scores[s, j] = canonical score of selected query s against row j. One warp per row; the row's share stays
// in registers/L1 while the warp walks the selected queries.
__global__ void dense_scores_kernel(const void* store, int dtype, int64_t n, int d, const void* q, int q_dtype,
                                    const int32_t* q_sel, int n_sel, int metric, float* out) {
    extern __shared__ __align__(16) float dq[];  // [n_sel_chunk, d4] staged queries
    const int lane = threadIdx.x & 31;
    const int d4 = ((d + 3) >> 2) << 2;
    const bool vec = (d % 4) == 0;
    const size_t esz = dtype == B2_F32 ? 4 : 2;
    const bool is_l2 = metric == B2_METRIC_L2;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    constexpr int QCHUNK = 8;
    for (int s0 = 0; s0 < n_sel; s0 += QCHUNK) {
        const int sc = min(QCHUNK, n_sel - s0);
        __syncthreads();
        for (int t = threadIdx.x; t < sc * d4; t += blockDim.x) {
            const int s = t / d4, i = t - s * d4;
            const int64_t qi = q_sel ? q_sel[s0 + s] : (s0 + s);
            dq[t] = i < d ? elem_f32(q, q_dtype, (size_t)qi * d + i) : 0.f;
        }
        __syncthreads();
        for (int64_t j = warp; j < n; j += nwarps) {
            const char* row = reinterpret_cast<const char*>(store) + (size_t)j * d * esz;
            for (int s = 0; s < sc; ++s) {
                const double part = is_l2 ? canonical_partial<true>(dq + s * d4, row, dtype, d, vec, lane)
                                          : canonical_partial<false>(dq + s * d4, row, dtype, d, vec, lane);
                const double tot = butterfly_sum(part);
                if (lane == 0) out[(size_t)(s0 + s) * n + j] = (float)tot;
            }
        }
    }
}

constexpr int SEL_THREADS = 512;
constexpr int SEL_MAX_K = 2048;

// ordered exclusive count of `flag` across the block (thread order), plus the block total
__device__ __forceinline__ int block_excl_count(bool flag, int* s_warp, int& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned b = __ballot_sync(FULL, flag);
    const int in_warp = __popc(b & ((1u << lane) - 1));
    __syncthreads();
    if (lane == 0) s_warp[warp] = __popc(b);
    __syncthreads();
    int before = 0, tot = 0;
    for (int w = 0; w < SEL_THREADS / 32; ++w) {
        const int cw = s_warp[w];
        before += w < warp ? cw : 0;
        tot += cw;
    }
    total = tot;
    return before + in_warp;
}

// One CTA per selected query: exact top-k of scores[s, 0..n) under faiss's heap rule.
__global__ void __launch_bounds__(SEL_THREADS)
dense_select_kernel(const float* scores, int64_t n, const int32_t* q_sel, int metric, int k, const int64_t* id_map,
                    int64_t id_offset, float* out_scores, int64_t* out_idx) {
    __shared__ int hist[256];
    __shared__ int s_warp[SEL_THREADS / 32];
    __shared__ uint32_t s_prefix, s_mask;
    __shared__ int s_kk, s_nbetter, s_nties;
    __shared__ uint64_t s_out[SEL_MAX_K];      // collected (key<<32 | tie-order id), later sorted
    __shared__ uint32_t s_ties[SEL_MAX_K];     // ids of the ties inside the first-k-by-id window, ascending
    const int s = blockIdx.x;
    const int64_t qo = q_sel ? q_sel[s] : s;
    const float* row = scores + (size_t)s * n;
    const bool is_l2 = metric == B2_METRIC_L2;
    const int tid = threadIdx.x;
    const int keff = (int)(n < k ? n : k);

    uint32_t vkey = 0xffffffffu;
    int r_keep = 0;
    if (n > k) {
        // radix select: the k-th smallest best-first key
        if (tid == 0) { s_prefix = 0; s_mask = 0; s_kk = k; }
        __syncthreads();
        for (int shift = 24; shift >= 0; shift -= 8) {
            for (int i = tid; i < 256; i += SEL_THREADS) hist[i] = 0;
            __syncthreads();
            const uint32_t prefix = s_prefix, mask = s_mask;
            for (int64_t j = tid; j < n; j += SEL_THREADS) {
                const uint32_t key = best_first_key(row[j], metric);
                if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255], 1);
            }
            __syncthreads();
            if (tid == 0) {
                int kk = s_kk, cum = 0, b = 0;
                for (b = 0; b < 256; ++b) {
                    if (cum + hist[b] >= kk) break;
                    cum += hist[b];
                }
                s_kk = kk - cum;
                s_prefix = prefix | ((uint32_t)b << shift);
                s_mask = mask | (0xffu << shift);
            }
            __syncthreads();
        }
        vkey = s_prefix;
        r_keep = s_kk;  // ties at vkey that belong to the top k
    }
    if (tid == 0) { s_nbetter = 0; s_nties = 0; }
    __syncthreads();

    // collect everything strictly better than v (unordered), and the ties inside the first k of S by id (ordered)
    int running_s = 0;
    for (int64_t base = 0; base < n; base += SEL_THREADS) {
        const int64_t j = base + tid;
        uint32_t key = 0xffffffffu;
        bool in_s = false, is_tie = false, better = false;
        if (j < n) {
            key = best_first_key(row[j], metric);
            if (n > k) {
                better = key < vkey;
                is_tie = key == vkey;
                in_s = better || is_tie;
            } else {
                better = true;
            }
        }
        if (better) {
            const int slot = atomicAdd(&s_nbetter, 1);
            const uint32_t tie = is_l2 ? (uint32_t)j : ~(uint32_t)j;
            if (slot < SEL_MAX_K) s_out[slot] = ((uint64_t)key << 32) | tie;
        }
        if (n > k && running_s < k) {  // running_s is block-uniform
            if (__syncthreads_or(in_s)) {
                int tot_s = 0;
                const int pos = running_s + block_excl_count(in_s, s_warp, tot_s);
                const bool tie_in_window = is_tie && pos < k;
                int tot_t = 0;
                const int tpos = block_excl_count(tie_in_window, s_warp, tot_t);
                const int tbase = s_nties;
                if (tie_in_window && tbase + tpos < SEL_MAX_K) s_ties[tbase + tpos] = (uint32_t)j;
                __syncthreads();
                if (tid == 0) s_nties = tbase + tot_t;
                running_s += tot_s;
                __syncthreads();
            }
        }
    }
    __syncthreads();
    const int c = s_nbetter;
    if (n > k) {
        const int t = s_nties;
        // L2: first r ties (ascending id). IP: the last r of the t window ties (e_{t-r+1} .. e_t).
        const int first = is_l2 ? 0 : t - r_keep;
        for (int i = tid; i < r_keep; i += SEL_THREADS) {
            const uint32_t id = s_ties[first + i];
            s_out[c + i] = ((uint64_t)vkey << 32) | (is_l2 ? id : ~id);
        }
    }
    // sort the keff collected entries (bitonic in shared memory, padded with worst keys)
    int npow = 1;
    while (npow < keff) npow <<= 1;
    __syncthreads();
    for (int i = keff + tid; i < npow; i += SEL_THREADS) s_out[i] = KEY_WORST;
    __syncthreads();
    for (int kk = 2; kk <= npow; kk <<= 1) {
        for (int j = kk >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < npow; i += SEL_THREADS) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const bool up = (i & kk) == 0;
                    const uint64_t a = s_out[i], b = s_out[ixj];
                    if ((a > b) == up) { s_out[i] = b; s_out[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
    const float pad = is_l2 ? FLT_MAX : -FLT_MAX;
    for (int o = tid; o < k; o += SEL_THREADS) {
        float sc = pad;
        int64_t oid = -1;
        if (o < keff) {
            const uint64_t kk2 = s_out[o];
            const uint32_t lo = (uint32_t)(kk2 & 0xffffffffu);
            const int64_t id = (int64_t)(is_l2 ? lo : ~lo);
            sc = best_first_unkey((uint32_t)(kk2 >> 32), metric);
            oid = id_map ? id_map[id] : id + id_offset;
        }
        out_scores[(size_t)qo * k + o] = sc;
        out_idx[(size_t)qo * k + o] = oid;
    }
}

// ---- large k (> SEL_MAX_K): full sort of dense score rows --------------------------------------------------------------------
// The cascade callers ask for K = len(df) (lotus/sem_ops/sem_filter.py:486-497, sem_join.py:343-373, sem_topk.py:782-788):
// every row is reported, best first. Keys (best-first score key << 32 | tie order) are built from the canonical scores, sorted
// by a device-wide radix sort (CUB — library code, a plumbing step here: the scores are ours), and the first k are unpacked.
// faiss switches to a reservoir for k >= 100 whose tie retention at the cut is unspecified; sorted truncation with the heap's
// order ((score desc, id desc) for IP, (dist asc, id asc) for L2) is used.
__global__ void dense_keys_kernel(const float* scores, int64_t n, int rows, int metric, uint64_t* keys) {
    const bool is_l2 = metric == B2_METRIC_L2;
    const int64_t total = (int64_t)rows * n;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j = t % n;
        keys[t] = ((uint64_t)best_first_key(scores[t], metric) << 32) | (is_l2 ? (uint32_t)j : ~(uint32_t)j);
    }
}

__global__ void dense_unpack_kernel(const uint64_t* keys, int64_t n, int rows, const int32_t* q_sel, int64_t q_base, int metric, int k,
                                    const int64_t* id_map, int64_t id_offset, float* out_scores, int64_t* out_idx) {
    const bool is_l2 = metric == B2_METRIC_L2;
    const float pad = is_l2 ? FLT_MAX : -FLT_MAX;
    const int64_t total = (int64_t)rows * k;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = t / k, o = t - s * k;
        const int64_t qo = q_sel ? (int64_t)q_sel[s] : q_base + s;
        float sc = pad;
        int64_t oid = -1;
        if (o < n) {
            const uint64_t e = keys[s * n + o];
            const uint32_t lo = (uint32_t)(e & 0xffffffffu);
            const int64_t id = (int64_t)(is_l2 ? lo : ~lo);
            sc = best_first_unkey((uint32_t)(e >> 32), metric);
            oid = id_map ? id_map[id] : id + id_offset;
        }
        out_scores[(size_t)qo * k + o] = sc;
        out_idx[(size_t)qo * k + o] = oid;
    }
}

struct RowOffset {
    int64_t n;
    __host__ __device__ int64_t operator()(int64_t i) const { return i * n; }
};

// ---- k-way merge of per-shard lists -----------------------------------------------------------------------------
template <int R>
__global__ void __launch_bounds__(128) merge_topk_kernel(const float* scores, const int64_t* idx, int g, int64_t nq, int k,
                                                         int metric, float* out_scores, int64_t* out_idx) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t q = blockIdx.x * 4LL + warp;
    if (q >= nq) return;
    const bool is_l2 = metric == B2_METRIC_L2;
    const int total = g * k;
    uint64_t keys[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int e = r * 32 + lane;
        uint64_t kk = KEY_WORST;
        if (e < total) {
            const int gi = e / k, pi = e - gi * k;
            const size_t off = ((size_t)gi * nq + q) * k + pi;
            if (idx[off] >= 0) {
                // equal scores: shard lists are already in faiss tie order; lower shards hold lower ids
                const uint32_t tie = is_l2 ? (uint32_t)e : (uint32_t)((g - 1 - gi) * k + pi);
                kk = ((uint64_t)best_first_key(scores[off], metric) << 32) | tie;
            }
        }
        keys[r] = kk;
    }
    warp_bitonic_sort<R>(keys, lane);
    const float pad = is_l2 ? FLT_MAX : -FLT_MAX;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int o = r * 32 + lane;
        if (o < k) {
            float sc = pad;
            int64_t oid = -1;
            if (keys[r] != KEY_WORST) {
                const uint32_t tie = (uint32_t)(keys[r] & 0xffffffffu);
                int gi, pi;
                if (is_l2) { gi = tie / k; pi = tie - gi * k; }
                else { const int gr = tie / k; pi = tie - gr * k; gi = g - 1 - gr; }
                const size_t off = ((size_t)gi * nq + q) * k + pi;
                sc = scores[off];
                oid = idx[off];
            }
            out_scores[(size_t)q * k + o] = sc;
            out_idx[(size_t)q * k + o] = oid;
        }
    }
}

// out[i] = canonical ||pts[i] - cent[assign[i]]||^2 (what kmeans.index.search(x, 1) reports for the winner). Warp per point.
__global__ void exact_l2_assigned_kernel(const void* pts, int dtype, int64_t m, int d, const float* cent, const int64_t* assign,
                                         float* out) {
    extern __shared__ __align__(16) float el_q[];  // [warps per block][d4]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int d4 = ((d + 3) >> 2) << 2;
    float* q_s = el_q + (size_t)wib * d4;
    const bool vec = (d % 4) == 0;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp; i < m; i += nwarps) {
        __syncwarp();
        for (int t = lane; t < d4; t += 32) q_s[t] = t < d ? elem_f32(pts, dtype, (size_t)i * d + t) : 0.f;
        __syncwarp();
        const int64_t c = assign[i];
        float r = FLT_MAX;
        if (c >= 0) {
            const double part = canonical_partial<true>(q_s, cent + (size_t)c * d, B2_F32, d, vec, lane);
            r = (float)butterfly_sum(part);
        }
        if (lane == 0) out[i] = r;
    }
}

// Row-sharded search, stage 1: lower[q] = (the j-th best filter score among this shard's candidates) - eps, a lower bound on the
// exact scores of j rows of this shard. After an all-reduce(MIN) over the ranks with j = ceil(k / ranks), ranks * j >= k rows of
// the index are known to score at least that much. Warp per query; up to 32 * LB_R candidate entries.
constexpr int LB_R = 32;
__global__ void shard_lower_bound_kernel(const float* cand_score, const int32_t* cand_id, int64_t nq, int n_lists, int list_len, int j,
                                         const float* qnorm2, float max_norm, float rel_eps, float abs_eps, const int32_t* q_bad,
                                         int metric, float* lower) {
    const int lane = threadIdx.x & 31;
    const int64_t q = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (q >= nq) return;
    if (q_bad && q_bad[q]) {  // no finite filter operand: no bound
        if (lane == 0) lower[q] = -INFINITY;
        return;
    }
    const int total = n_lists * list_len;
    float v[LB_R];
#pragma unroll
    for (int r = 0; r < LB_R; ++r) {
        const int e = r * 32 + lane;
        float s = -INFINITY;
        if (e < total) {
            const size_t off = (size_t)q * total + e;
            if (cand_id[off] >= 0) s = cand_score[off];
        }
        v[r] = s;
    }
    float tj = -INFINITY;
    for (int t = 0; t < j; ++t) {
        float m = v[0];
#pragma unroll
        for (int r = 1; r < LB_R; ++r) m = fmaxf(m, v[r]);
        float M = m;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) M = fmaxf(M, __shfl_xor_sync(FULL, M, off));
        tj = M;
        if (!(M > -INFINITY)) break;  // fewer than j candidates (or NaN): no bound
        const unsigned owners = __ballot_sync(FULL, m == M);
        if (lane == __ffs(owners) - 1) {  // remove ONE instance of the maximum
            bool done = false;
#pragma unroll
            for (int r = 0; r < LB_R; ++r)
                if (!done && v[r] == M) {
                    v[r] = -INFINITY;
                    done = true;
                }
        }
    }
    if (lane == 0) {
        float out = -INFINITY;
        if (tj > -INFINITY) {
            const double qn = sqrt((double)qnorm2[q]), mx = (double)max_norm;
            const double ip_err = filter_ip_err((double)rel_eps, (double)abs_eps, qn, mx);
            const double eps = metric == B2_METRIC_L2 ? 2.0 * ip_err + 2.4e-7 * (mx * mx + 2.0 * qn * mx) + 1.3e-7 * qn * qn + 1e-30
                                                      : ip_err * (1.0 + 1.3e-7) + 1e-30;
            out = (float)((double)tj - eps - 4.8e-7 * fabs((double)tj));
        }
        lower[q] = out;
    }
}

__global__ void fill_f32_kernel(float* p, int64_t n, float v) {
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) p[t] = v;
}

int grid_for(int64_t work_items, int threads, int cap = 148 * 16) {
    int64_t g = ceil_div(work_items, threads);
    if (g < 1) g = 1;
    return (int)std::min<int64_t>(g, cap);
}

}  // namespace

int dense_max_k() { return 1 << 24; }
int dense_select_max_k() { return SEL_MAX_K; }

int launch_prep_queries(const void* q, int q_dtype, int64_t nq, int d, void* q_filt, int filt_dtype,
                        int64_t filt_pitch, cudaStream_t stream, int32_t* bad) {
    if (nq <= 0) return B2_OK;
    prep_queries_kernel<<<grid_for(nq * filt_pitch, 256), 256, 0, stream>>>(q, q_dtype, nq, d, q_filt, filt_dtype, filt_pitch, bad);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

int launch_row_norms(const void* x, int dtype, int64_t n, int d, float* norm2, float* max_norm_dev, cudaStream_t stream) {
    B2_CUDA(cudaMemsetAsync(max_norm_dev, 0, sizeof(float), stream));
    if (n <= 0) return B2_OK;
    row_norms_kernel<<<grid_for(n * 32, 256), 256, 0, stream>>>(x, dtype, n, d, norm2, max_norm_dev);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

int shard_lower_bound_max_entries() { return 32 * LB_R; }

int launch_shard_lower_bound(const float* cand_score, const int32_t* cand_id, int64_t nq, int n_lists, int list_len, int j, const float* qnorm2,
                             float max_norm, float rel_eps, float abs_eps, const int32_t* q_bad, int metric, float* lower,
                             cudaStream_t stream) {
    if (nq <= 0) return B2_OK;
    shard_lower_bound_kernel<<<(unsigned)ceil_div(nq * 32, 128), 128, 0, stream>>>(cand_score, cand_id, nq, n_lists, list_len, j, qnorm2, max_norm,
                                                                                  rel_eps, abs_eps, q_bad, metric, lower);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

int launch_fill_f32(float* p, int64_t n, float v, cudaStream_t stream) {
    if (n <= 0) return B2_OK;
    fill_f32_kernel<<<grid_for(n, 256), 256, 0, stream>>>(p, n, v);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

int launch_exact_l2_assigned(const void* pts, int dtype, int64_t m, int d, const float* cent, const int64_t* assign, float* out,
                             cudaStream_t stream) {
    if (m <= 0) return B2_OK;
    const int d4 = ((d + 3) >> 2) << 2;
    const size_t smem = (size_t)8 * d4 * 4;
    if (smem > 200 * 1024) {
        set_error("embedding dimension %d too large for the exact distance kernel", d);
        return B2_ERANGE;
    }
    if (smem > 48 * 1024) B2_CUDA(cudaFuncSetAttribute(exact_l2_assigned_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    exact_l2_assigned_kernel<<<grid_for(m * 32, 256, 148 * 8), 256, smem, stream>>>(pts, dtype, m, d, cent, assign, out);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

int launch_convert_pad(const void* x, int dtype, int64_t n, int d, void* out, int out_dtype, int64_t out_pitch,
                       cudaStream_t stream, int32_t* bad) {
    if (n <= 0) return B2_OK;
    convert_pad_kernel<<<grid_for(n * out_pitch, 256), 256, 0, stream>>>(x, dtype, n, d, out, out_dtype, out_pitch, bad);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

int launch_gather_rows(const void* x, int dtype, int d, const int64_t* ids, int64_t m, int64_t n, void* out,
                       int* err_flag, cudaStream_t stream) {
    if (m <= 0) return B2_OK;
    const size_t row_bytes = (size_t)d * (dtype == B2_F32 ? 4 : 2);
    gather_rows_kernel<<<grid_for(m * 32, 256), 256, 0, stream>>>(reinterpret_cast<const char*>(x), row_bytes, ids, m, n,
                                                                  reinterpret_cast<char*>(out), err_flag);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

template <int R>
static int launch_finalize_r(const FinalizeParams& p, cudaStream_t stream) {
    const int d4 = ((p.d + 3) >> 2) << 2;
    const size_t smem = (size_t)FIN_WARPS * ((size_t)d4 * 4 + (size_t)(32 * R) * 16);
    auto kern = finalize_kernel<R>;
    if (smem > 48 * 1024) {
        if (smem > 200 * 1024) {
            set_error("embedding dimension %d too large for the finalize kernel", p.d);
            return B2_ERANGE;
        }
        B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    kern<<<(unsigned)ceil_div(p.nq, FIN_WARPS), FIN_WARPS * 32, smem, stream>>>(p);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

int launch_finalize(const MatView& X, const void* q, int q_dtype, int64_t nq, int metric, int k, int kp, int list_len,
                    int n_splits, const float* cand_score, const int32_t* cand_id, const float* cand_thr,
                    float rel_eps, const int64_t* id_map, int64_t id_offset, float* out_scores, int64_t* out_idx,
                    int32_t* flags, int32_t* sel, int32_t* sel_count, cudaStream_t stream, const float* hint,
                    const int32_t* q_bad) {
    if (nq <= 0) return B2_OK;
    FinalizeParams p;
    p.hint = hint;
    p.q_bad = q_bad;
    p.abs_eps = filter_abs_eps(X.dtype, X.filt_dtype, q_dtype, X.d);
    p.sel = sel;
    p.sel_count = sel_count;
    p.store = X.store;
    p.q = q;
    p.cand_score = cand_score;
    p.cand_id = cand_id;
    p.cand_thr = cand_thr;
    p.id_map = id_map;
    p.out_scores = out_scores;
    p.out_idx = out_idx;
    p.flags = flags;
    p.nq = nq;
    p.id_offset = id_offset;
    p.d = X.d;
    p.dtype = X.dtype;
    p.q_dtype = q_dtype;
    p.metric = metric;
    p.k = k;
    p.kp = kp;
    p.list_len = list_len;
    p.n_splits = n_splits;
    p.rel_eps = rel_eps;
    p.max_norm = X.max_norm;
    p.max_norm_dev = X.max_norm_dev;
    g_stats[ST_RESCORED] += nq * (int64_t)kp;
    // survivors kept through the merge: the filter's list capacity for k <= 64; k + 32 when several splits share a large k
    // (the 32 extra by-filter-score candidates are what the prune / certificate margins need)
    const int need = std::max(kp, k > 64 ? std::min(k + 32, 1024) : 0);
    if (need <= 32) return launch_finalize_r<1>(p, stream);
    if (need <= 64) return launch_finalize_r<2>(p, stream);
    if (need <= 128) return launch_finalize_r<4>(p, stream);
    if (need <= 256) return launch_finalize_r<8>(p, stream);
    if (need <= 512) return launch_finalize_r<16>(p, stream);
    if (need <= 1024) return launch_finalize_r<32>(p, stream);
    set_error("internal: finalize capacity %d", need);
    return B2_EINVAL;
}

// workspace bytes the full-sort path needs for `rows` score rows of length n: keys in + keys out + the sort's scratch
size_t dense_sort_ws_bytes(int64_t rows, int64_t n) {
    const size_t items = (size_t)rows * (size_t)n;
    size_t temp = 0;
    if (rows <= 4) {
        cub::DeviceRadixSort::SortKeys(nullptr, temp, (const uint64_t*)nullptr, (uint64_t*)nullptr, (int64_t)n);
    } else {
        cub::CountingInputIterator<int64_t> cnt(0);
        cub::TransformInputIterator<int64_t, RowOffset, cub::CountingInputIterator<int64_t>> beg(cnt, RowOffset{n});
        cub::DeviceSegmentedSort::SortKeys(nullptr, temp, (const uint64_t*)nullptr, (uint64_t*)nullptr, (int64_t)items, (int64_t)rows, beg, beg + 1);
    }
    return 2 * items * sizeof(uint64_t) + temp + 512;
}

int launch_dense_topk(const MatView& X, const void* q, int q_dtype, int64_t nq, const int32_t* q_sel, int64_t n_sel,
                      int metric, int k, const int64_t* id_map, int64_t id_offset, float* dense_ws,
                      int64_t dense_ws_rows, uint64_t* sort_ws, float* out_scores, int64_t* out_idx, cudaStream_t stream) {
    (void)nq;
    if (n_sel <= 0) return B2_OK;
    const bool full_sort = k > SEL_MAX_K;  // needs sort_ws of dense_sort_ws_bytes(dense_ws_rows, n)
    if (full_sort && !sort_ws) {
        set_error("internal: k=%d needs the sort workspace", k);
        return B2_EINVAL;
    }
    const int d4 = ((X.d + 3) >> 2) << 2;
    const size_t smem = (size_t)8 * d4 * 4;
    if (smem > 48 * 1024) {
        if (smem > 200 * 1024) {
            set_error("embedding dimension %d too large for the dense path", X.d);
            return B2_ERANGE;
        }
        B2_CUDA(cudaFuncSetAttribute(dense_scores_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    for (int64_t s0 = 0; s0 < n_sel; s0 += dense_ws_rows) {
        const int sc = (int)std::min<int64_t>(dense_ws_rows, n_sel - s0);
        const int32_t* sel = q_sel ? q_sel + s0 : nullptr;
        // without a selection list the batch is the contiguous query range [s0, s0+sc)
        const void* qb = q_sel ? q : reinterpret_cast<const char*>(q) + (size_t)s0 * X.d * (q_dtype == B2_F32 ? 4 : 2);  // bf16, fp16: 2
        if (X.n > 0) {
            dense_scores_kernel<<<grid_for(X.n * 32, 256, 148 * 8), 256, smem, stream>>>(X.store, X.dtype, X.n, X.d, qb, q_dtype,
                                                                                       sel, sc, metric, dense_ws);
            B2_LAUNCH_CHECK();
        }
        if (full_sort) {
            const size_t items = (size_t)sc * (size_t)X.n;
            uint64_t* k_in = sort_ws;
            uint64_t* k_out = sort_ws + (size_t)dense_ws_rows * X.n;
            void* temp = k_out + (size_t)dense_ws_rows * X.n;
            size_t temp_bytes = dense_sort_ws_bytes(dense_ws_rows, X.n) - 2 * (size_t)dense_ws_rows * X.n * sizeof(uint64_t) - 512;
            if (X.n > 0) {
                dense_keys_kernel<<<grid_for((int64_t)items, 256), 256, 0, stream>>>(dense_ws, X.n, sc, metric, k_in);
                B2_LAUNCH_CHECK();
                if (dense_ws_rows <= 4) {
                    for (int r = 0; r < sc; ++r)
                        B2_CUDA(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, k_in + (size_t)r * X.n, k_out + (size_t)r * X.n, (int64_t)X.n,
                                                              0, 64, stream));
                } else {
                    cub::CountingInputIterator<int64_t> cnt(0);
                    cub::TransformInputIterator<int64_t, RowOffset, cub::CountingInputIterator<int64_t>> beg(cnt, RowOffset{X.n});
                    B2_CUDA(cub::DeviceSegmentedSort::SortKeys(temp, temp_bytes, k_in, k_out, (int64_t)items, (int64_t)sc, beg, beg + 1, stream));
                }
                g_stats[ST_LAUNCHES]++;
            }
            dense_unpack_kernel<<<grid_for((int64_t)sc * k, 256), 256, 0, stream>>>(k_out, X.n, sc, sel, s0, metric, k, id_map, id_offset,
                                                                                  out_scores, out_idx);
            B2_LAUNCH_CHECK();
        } else {
            float* os = q_sel ? out_scores : out_scores + (size_t)s0 * k;
            int64_t* oi = q_sel ? out_idx : out_idx + (size_t)s0 * k;
            dense_select_kernel<<<sc, SEL_THREADS, 0, stream>>>(dense_ws, X.n, sel, metric, k, id_map, id_offset, os, oi);
            B2_LAUNCH_CHECK();
        }
    }
    return B2_OK;
}

int launch_merge_topk(const float* scores, const int64_t* idx, int g, int64_t nq, int k, int metric, float* out_scores,
                      int64_t* out_idx, cudaStream_t stream) {
    if (nq <= 0) return B2_OK;
    const int total = g * k;
    const unsigned grid = (unsigned)ceil_div(nq, 4);
#define B2_MERGE_CASE(RR)                                                                                        \
    if (total <= 32 * RR) {                                                                                      \
        merge_topk_kernel<RR><<<grid, 128, 0, stream>>>(scores, idx, g, nq, k, metric, out_scores, out_idx);     \
        B2_LAUNCH_CHECK();                                                                                       \
        return B2_OK;                                                                                            \
    }
    B2_MERGE_CASE(1)
    B2_MERGE_CASE(2)
    B2_MERGE_CASE(4)
    B2_MERGE_CASE(8)
    B2_MERGE_CASE(16)
    B2_MERGE_CASE(32)
#undef B2_MERGE_CASE
    set_error("merge of %d lists x k=%d exceeds 1024 candidates per query", g, k);
    return B2_ERANGE;
}


namespace {

// ---- packed (score, local id) lists for the row-sharded exchange: 8 bytes per entry instead of 12 --------------------------
__global__ void pack_topk_kernel(const float* scores, const int64_t* idx, int64_t total, uint64_t* out) {
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t id = idx[t];
        out[t] = ((uint64_t)__float_as_uint(scores[t]) << 32) | (id < 0 ? 0xffffffffu : (uint32_t)id);
    }
}

template <int R>
__global__ void __launch_bounds__(128) merge_packed_kernel(const uint64_t* packed, MergeOffsets offs, int g, int64_t nq, int k, int metric,
                                                           float* out_scores, int64_t* out_idx) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t q = blockIdx.x * 4LL + warp;
    if (q >= nq) return;
    const bool is_l2 = metric == B2_METRIC_L2;
    const int total = g * k;
    uint64_t keys[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int e = r * 32 + lane;
        uint64_t kk = KEY_WORST;
        if (e < total) {
            const int gi = e / k, pi = e - gi * k;
            const uint64_t ent = packed[((size_t)gi * nq + q) * k + pi];
            if ((uint32_t)ent != 0xffffffffu) {
                // equal scores: shard lists are already in faiss tie order; lower shards hold lower ids
                const uint32_t tie = is_l2 ? (uint32_t)e : (uint32_t)((g - 1 - gi) * k + pi);
                kk = ((uint64_t)best_first_key(__uint_as_float((uint32_t)(ent >> 32)), metric) << 32) | tie;
            }
        }
        keys[r] = kk;
    }
    warp_bitonic_sort<R>(keys, lane);
    const float pad = is_l2 ? FLT_MAX : -FLT_MAX;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int o = r * 32 + lane;
        if (o < k) {
            float sc = pad;
            int64_t oid = -1;
            if (keys[r] != KEY_WORST) {
                const uint32_t tie = (uint32_t)(keys[r] & 0xffffffffu);
                int gi, pi;
                if (is_l2) { gi = tie / k; pi = tie - gi * k; }
                else { const int gr = tie / k; pi = tie - gr * k; gi = g - 1 - gr; }
                const uint64_t ent = packed[((size_t)gi * nq + q) * k + pi];
                sc = __uint_as_float((uint32_t)(ent >> 32));
                oid = (int64_t)(uint32_t)ent + offs.v[gi];
            }
            out_scores[(size_t)q * k + o] = sc;
            out_idx[(size_t)q * k + o] = oid;
        }
    }
}

}  // namespace

int launch_pack_topk(const float* scores, const int64_t* idx, int64_t total, uint64_t* out, cudaStream_t stream) {
    if (total <= 0) return B2_OK;
    pack_topk_kernel<<<grid_for(total, 256), 256, 0, stream>>>(scores, idx, total, out);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

int launch_merge_packed(const uint64_t* packed, const int64_t* shard_offsets, int g, int64_t nq, int k, int metric, float* out_scores,
                        int64_t* out_idx, cudaStream_t stream) {
    if (nq <= 0) return B2_OK;
    if (g > MergeOffsets::MAX) {
        set_error("merge of %d shards: at most %d", g, MergeOffsets::MAX);
        return B2_ERANGE;
    }
    MergeOffsets offs;
    for (int i = 0; i < g; ++i) offs.v[i] = shard_offsets[i];
    const int total = g * k;
    const unsigned grid = (unsigned)ceil_div(nq, 4);
#define B2_MERGEP_CASE(RR)                                                                                              \
    if (total <= 32 * RR) {                                                                                            \
        merge_packed_kernel<RR><<<grid, 128, 0, stream>>>(packed, offs, g, nq, k, metric, out_scores, out_idx);        \
        B2_LAUNCH_CHECK();                                                                                             \
        return B2_OK;                                                                                                  \
    }
    B2_MERGEP_CASE(1)
    B2_MERGEP_CASE(2)
    B2_MERGEP_CASE(4)
    B2_MERGEP_CASE(8)
    B2_MERGEP_CASE(16)
    B2_MERGEP_CASE(32)
#undef B2_MERGEP_CASE
    set_error("merge of %d lists x k=%d exceeds 1024 candidates per query", g, k);
    return B2_ERANGE;
}

}  // namespace b2
