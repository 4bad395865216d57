// common.cuh — shared declarations for libb2lotus.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>

#include "../../include/lotus_b200.h"

namespace b2 {

// ---- error plumbing ------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
extern int64_t g_stats[8];
enum { ST_LAUNCHES = 0, ST_QUERIES = 1, ST_FALLBACK = 2, ST_FILTER_LAUNCHES = 3, ST_RESCORED = 4, ST_SECOND_LEVEL = 5 };

#define B2_CUDA(expr)                                                                              \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            b2::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return B2_ECUDA;                                                                       \
        }                                                                                          \
    } while (0)

#define B2_LAUNCH_CHECK()                                                                          \
    do {                                                                                           \
        b2::g_stats[b2::ST_LAUNCHES]++;                                                            \
        cudaError_t _e = cudaGetLastError();                                                       \
        if (_e != cudaSuccess) {                                                                   \
            b2::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
            return B2_ECUDA;                                                                       \
        }                                                                                          \
    } while (0)

#define B2_TRY(expr)            \
    do {                        \
        int _rc = (expr);       \
        if (_rc != B2_OK) return _rc; \
    } while (0)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

// ---- order-preserving keys --------------------------------------------------------------------------------
// ord(f) is monotone in f (for non-NaN f); -0.0 is folded onto +0.0 first.
__host__ __device__ __forceinline__ uint32_t f32_ord(float f) {
    f = f + 0.0f;
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    uint32_t u;
    memcpy(&u, &f, 4);
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float f32_unord(uint32_t k) {
    uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    float f;
    memcpy(&f, &u, 4);
    return f;
#endif
}
// "best first when sorted ascending": IP wants large scores first, L2 small distances first.
__host__ __device__ __forceinline__ uint32_t best_first_key(float s, int metric) {
    uint32_t o = f32_ord(s);
    return metric == B2_METRIC_IP ? ~o : o;
}
__host__ __device__ __forceinline__ float best_first_unkey(uint32_t k, int metric) {
    return f32_unord(metric == B2_METRIC_IP ? ~k : k);
}

// ---- a matrix the kernels can search ---------------------------------------------------------------------
// `store` holds the exact values (dtype f32, bf16 or f16, row pitch `d`). `filt` is what the tcgen05 filter
// streams through TMA: bf16 / fp16 (pitch multiple of 8 elements) for a bf16 / fp16 index, fp32 (pitch multiple of 4)
// read as TF32 for an fp32 index; it aliases `store` whenever the pitch already qualifies.
struct MatView {
    const void* store = nullptr;
    const void* filt = nullptr;
    const float* norm2 = nullptr;  // [n] fp32 squared norms of the exact rows (L2 filter epilogue)
    int64_t n = 0;
    int32_t d = 0;
    int32_t dtype = B2_F32;       // element type of `store`
    int32_t filt_dtype = B2_F32;  // element type of `filt`: B2_BF16 / B2_F16 -> kind::f16 MMA, B2_F32 -> kind::tf32 MMA
    int64_t filt_pitch = 0;  // elements
    // fp32 stores only (optional): a bf16 rounding of the rows, pitch multiple of 8. When present, searches run a FIRST level on it
    // (kind::f16 at twice the tf32 rate, operand error 2^-8 per fp32 operand in the certificate) and only the queries whose
    // certificate fails there go through the tf32 filter on `filt`.
    const void* filt16 = nullptr;
    int64_t filt16_pitch = 0;
    float max_norm = 0.f;    // max_j ||x_j|| (upper bound), for the certification margin
    const float* max_norm_dev = nullptr;  // when set, the kernels read the bound from device memory instead (no host sync:
                                          // the k-means loop rebuilds its centroid view every iteration)
};

struct SearchWorkspace;

// ---- certificate margins (api.cu) -----------------------------------------------------------------------------
// |filter inner product - exact inner product| <= rel ||q|| ||x|| + abs (||q|| + ||x|| + abs), rel = filter_rel_eps(...),
// abs = filter_abs_eps(...) (non-zero only when an fp32 / bf16 operand is rounded to fp16, whose subnormals lose bits)
float filter_rel_eps(int store_dtype, int filt_dtype, int q_dtype, int d);
float filter_abs_eps(int store_dtype, int filt_dtype, int q_dtype, int d);
__host__ __device__ __forceinline__ double filter_ip_err(double rel, double abs_eps, double qn, double xn) {
    return rel * qn * xn + abs_eps * (qn + xn + abs_eps);
}

// ---- kernels / launchers (one per .cu) ------------------------------------------------------------------
// knn_filter_sm100.cu
int filter_kp_for_k(int k);  // candidate-list capacity used for a given k, 0 = k too large for the filter
int launch_knn_filter(const MatView& X, const void* q_filt, int64_t q_pitch, int64_t nq, int metric, int kp,
                      int n_splits, bool two_cta, float* cand_score, int32_t* cand_id, float* cand_thr, int device,
                      cudaStream_t stream, bool top1 = false, int units_whole = 0);
bool filter_use_pair(int64_t nq);
int filter_choose_splits(int64_t nq, int64_t n, int num_sms, bool two_cta, bool top1 = false, int min_splits = 1,
                         int* units_whole = nullptr);  // 0: impossible; *units_whole > 0: two-phase schedule (see the definition)
int filter_min_splits_for_k(int k);
int launch_pair_filter(const MatView& X, float thr, int part, int nparts, int32_t* pair_i, int32_t* pair_j,
                       unsigned long long* pair_count, unsigned long long cap, int device, cudaStream_t stream);

// knn_exact.cu
// bad (nullable, [nq], zeroed by the caller): set to 1 for a query with an element that is not a finite filter operand (beyond
// fp16's range when filt_dtype == B2_F16); its filter row is written with a zero there and finalize sends it to the exact path
int launch_prep_queries(const void* q, int q_dtype, int64_t nq, int d, void* q_filt, int filt_dtype,
                        int64_t filt_pitch, cudaStream_t stream, int32_t* bad = nullptr);
int launch_row_norms(const void* x, int dtype, int64_t n, int d, float* norm2, float* max_norm_dev,
                     cudaStream_t stream);
// bad (nullable): set to 1 when an fp16 output element is not finite (it is written as 0)
int launch_convert_pad(const void* x, int dtype, int64_t n, int d, void* out, int out_dtype, int64_t out_pitch,
                       cudaStream_t stream, int32_t* bad = nullptr);
int launch_exact_l2_assigned(const void* pts, int dtype, int64_t m, int d, const float* cent, const int64_t* assign, float* out,
                             cudaStream_t stream);
int launch_gather_rows(const void* x, int dtype, int d, const int64_t* ids, int64_t m, int64_t n, void* out,
                       int* err_flag, cudaStream_t stream);
int launch_finalize(const MatView& X, const void* q, int q_dtype, int64_t nq, int metric, int k, int kp, int list_len,
                    int n_lists, const float* cand_score, const int32_t* cand_id, const float* cand_thr,
                    float rel_eps, const int64_t* id_map, int64_t id_offset, float* out_scores, int64_t* out_idx,
                    int32_t* flags, int32_t* sel, int32_t* sel_count, cudaStream_t stream, const float* hint = nullptr,
                    const int32_t* q_bad = nullptr);
int shard_lower_bound_max_entries();
int launch_shard_lower_bound(const float* cand_score, const int32_t* cand_id, int64_t nq, int n_lists, int list_len, int j, const float* qnorm2,
                             float max_norm, float rel_eps, float abs_eps, const int32_t* q_bad, int metric, float* lower,
                             cudaStream_t stream);
int launch_fill_f32(float* p, int64_t n, float v, cudaStream_t stream);
int launch_dense_topk(const MatView& X, const void* q, int q_dtype, int64_t nq, const int32_t* q_sel,
                      int64_t n_sel, int metric, int k, const int64_t* id_map, int64_t id_offset, float* dense_ws,
                      int64_t dense_ws_rows, uint64_t* sort_ws, float* out_scores, int64_t* out_idx, cudaStream_t stream);
int launch_merge_topk(const float* scores, const int64_t* idx, int g, int64_t nq, int k, int metric,
                      float* out_scores, int64_t* out_idx, cudaStream_t stream);
size_t dense_sort_ws_bytes(int64_t rows, int64_t n);  // workspace of the full-sort path for `rows` score rows
int launch_pack_topk(const float* scores, const int64_t* idx, int64_t total, uint64_t* out, cudaStream_t stream);
int launch_merge_packed(const uint64_t* packed, const int64_t* shard_offsets, int g, int64_t nq, int k, int metric, float* out_scores,
                        int64_t* out_idx, cudaStream_t stream);
int dense_max_k();         // largest k any path supports
int dense_select_max_k();  // largest k of the radix-select path (beyond it: full row sort)

}  // namespace b2
