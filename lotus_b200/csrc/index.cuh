// index.cuh — the b2_index handle and the pieces of the search pipeline shared by api.cu, dedup.cu, kmeans.cu.
#pragma once
#include <algorithm>

#include "common.cuh"

namespace b2 {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return B2_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error("cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
            p = nullptr;
            return B2_ENOMEM;
        }
        cap = want;
        return B2_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T>
    T* as() { return reinterpret_cast<T*>(p); }
};

struct HostBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return B2_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMallocHost(&p, bytes + 256);
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error("cudaMallocHost(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
            return B2_ENOMEM;
        }
        cap = bytes + 256;
        return B2_OK;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

struct KmWork;                 // kmeans.cu: per-handle k-means workspaces
void km_work_free(KmWork* w);  // (defined in kmeans.cu)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

}  // namespace b2

struct b2_index {
    using DevBuf = b2::DevBuf;
    using HostBuf = b2::HostBuf;
    using MatView = b2::MatView;
    int device = 0;
    int64_t n = 0;
    int32_t d = 0;
    int32_t dtype = B2_F32;
    int32_t metric = B2_METRIC_IP;
    DevBuf store, filt_pad, filt16, norm2, scalar;
    MatView view;
    // per-call workspaces
    DevBuf q_in, q_filt, cand_score, cand_id, cand_thr, flags, sel, dense, out_sc, out_id, ids_dev;
    DevBuf sub_store, sub_filt, sub_filt16, sub_norm2, sort_keys;
    DevBuf defer, q_sub, sub_sc, sub_id;  // two-level search of fp32 indexes: deferred queries, their rows and results
    HostBuf h_flags;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    float last_filter_ms = -1.f;
    b2::KmWork* km = nullptr;
    // row-sharded search in two stages (b2_index_search_stage1_dev / _stage2_packed_dev): what stage 1 left for stage 2
    struct Staged {
        bool active = false, filtered = false;  // filtered: the candidate lists of (q, nq, k) are in the workspace
        const void* q = nullptr;
        int64_t nq = 0;
        int32_t q_dtype = 0, k = 0, kp = 0, n_splits = 0;
        float rel_eps = 0.f, abs_eps = 0.f;
        bool q_bad = false;  // idx->q_bad holds the queries prep_queries flagged (fp16 filter operands)
    } staged;
    DevBuf q_norm2, q_bad;
};

namespace b2 {

static inline size_t esize(int dtype) { return dtype == B2_F32 ? 4 : 2; }  // B2_BF16, B2_F16: 2 bytes

// searchable view (filter operand, row norms, max norm) of a row-major device matrix
int build_view(const void* store, int64_t n, int d, int dtype, DevBuf& filt_pad, DevBuf& norm2, DevBuf& scalar, MatView& v,
               cudaStream_t st, DevBuf* filt16 = nullptr);
// the exact top-k pipeline on device buffers: tcgen05 filter -> finalize/certify -> dense fallback
int search_core(b2_index* idx, const MatView& X, int metric, const void* q_dev, int q_dtype, int64_t nq, int k,
                const int64_t* id_map, int64_t id_offset, float* out_sc, int64_t* out_id, cudaStream_t st, int level = 0);
float filter_rel_eps(int store_dtype, int filt_dtype, int q_dtype, int d);

}  // namespace b2
