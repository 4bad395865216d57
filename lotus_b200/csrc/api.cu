// api.cu — the C-ABI of libb2lotus.so (include/lotus_b200.h): handles, workspaces and the search pipeline
//   prep queries -> tcgen05 filter (knn_filter_sm100.cu) -> finalize/certify (knn_exact.cu) -> dense exact
//   fallback for uncertified queries.
// Reference call sites replaced: lotus/vector_store/faiss_vs.py:22-77 (see the header for the mapping).
#include <algorithm>
#include <cstring>
#include <atomic>
#include <mutex>
#include <thread>
#include <vector>

#include "index.cuh"

namespace b2 {

static thread_local std::string g_err;
int64_t g_stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
}

}  // namespace b2

using namespace b2;

namespace b2 {

// Build the searchable view of a row-major matrix that already sits in device memory.
int build_view(const void* store, int64_t n, int d, int dtype, DevBuf& filt_pad, DevBuf& norm2, DevBuf& scalar,
                      MatView& v, cudaStream_t st, DevBuf* filt16) {
    v.store = store;
    v.n = n;
    v.d = d;
    v.dtype = dtype;
    v.filt_dtype = dtype;
    const int align = dtype == B2_F32 ? 4 : 8;  // TMA row pitch must be a multiple of 16 bytes
    if (d % align == 0) {
        v.filt = store;
        v.filt_pitch = d;
    } else {
        v.filt_pitch = round_up(d, align);
        B2_TRY(filt_pad.ensure((size_t)std::max<int64_t>(n, 1) * v.filt_pitch * esize(dtype)));
        B2_TRY(launch_convert_pad(store, dtype, n, d, filt_pad.p, dtype, v.filt_pitch, st));
        v.filt = filt_pad.p;
    }
    v.filt16 = nullptr;
    v.filt16_pitch = 0;
    static const bool bf16_first = [] { const char* e = getenv("B2_F32_BF16_FIRST"); return e ? atoi(e) != 0 : true; }();
    if (filt16 && dtype == B2_F32 && bf16_first && n >= 4096) {
        v.filt16_pitch = round_up(d, 8);
        B2_TRY(filt16->ensure((size_t)n * v.filt16_pitch * 2));
        B2_TRY(launch_convert_pad(store, dtype, n, d, filt16->p, B2_BF16, v.filt16_pitch, st));
        v.filt16 = filt16->p;
    }
    B2_TRY(norm2.ensure((size_t)std::max<int64_t>(n, 1) * sizeof(float)));
    B2_TRY(scalar.ensure(64));
    B2_TRY(launch_row_norms(store, dtype, n, d, norm2.as<float>(), scalar.as<float>(), st));
    float mx = 0.f;
    B2_CUDA(cudaMemcpyAsync(&mx, scalar.p, sizeof(float), cudaMemcpyDeviceToHost, st));
    B2_CUDA(cudaStreamSynchronize(st));
    v.norm2 = norm2.as<float>();
    v.max_norm = mx;
    return B2_OK;
}

// relative (to ||q||*||x||) bound on |filter score - exact score| of the inner product
float filter_rel_eps(int store_dtype, int filt_dtype, int q_dtype, int d) {
    // fp32 accumulation inside the tensor core: products are exact, every accumulation step may lose one
    // (truncated) ulp of the running magnitude; (d + 64) * 2^-23 is generous. Exercised by tests/test_gpu_search.py and
    // tests/test_gpu_fuzz.py: a too-small bound shows up as a wrong neighbour, a too-large one only as fallback work.
    const double acc = (double)(d + 64) * 1.1920929e-7;
    double ex = 0.0, eq = 0.0;  // relative representation error of the corpus / query operand seen by the MMA
    if (filt_dtype == B2_F32) {  // kind::tf32 keeps 10 explicit mantissa bits of an fp32 operand
        ex = store_dtype == B2_F32 ? 9.765625e-4 : 0.0;  // bf16 and fp16 values (subnormals included) are exact in tf32
        eq = q_dtype == B2_F32 ? 9.765625e-4 : 0.0;
    } else if (filt_dtype == B2_F16) {  // kind::f16 on fp16 operands: 11 significant bits, exponents 2^-14 .. 2^15
        // fp32 rounded to fp16: 2^-11 relative in the normal range (the subnormal range is filter_abs_eps's). A bf16 value
        // (8 significant bits) in the normal range is exact; beyond the finite range prep_queries flags the query.
        ex = store_dtype == B2_F32 ? 4.8828125e-4 : 0.0;
        eq = q_dtype == B2_F32 ? 4.8828125e-4 : 0.0;
    } else {  // kind::f16 on bf16 operands
        ex = store_dtype == B2_F32 ? 3.90625e-3 : 0.0;  // fp32 values rounded to bf16 for the filter
        eq = q_dtype != B2_BF16 ? 3.90625e-3 : 0.0;     // fp32 and fp16 queries rounded to bf16 (fp16's range lies inside bf16's)
    }
    return (float)(acc + ex + eq + ex * eq + 1e-6);
}

// Absolute part of the bound: an operand rounded to fp16 from a type with a wider exponent range (fp32, bf16) may land in
// fp16's subnormal range, where the rounding error is up to 2^-25 per element whatever the value: 2^-25 sqrt(d) in norm.
// With ||dq|| <= eq ||q|| + a and ||dx|| <= ex ||x|| + a (a = this value, 0.1 % above 2^-25 sqrt(d) so that the eq a, ex a
// cross terms are inside it) the inner product moves by at most
//     rel_eps ||q|| ||x||  +  a (||q|| + ||x|| + a).
float filter_abs_eps(int store_dtype, int filt_dtype, int q_dtype, int d) {
    if (filt_dtype != B2_F16 || (store_dtype == B2_F16 && q_dtype == B2_F16)) return 0.f;
    return (float)(1.001 * 2.98023223876953125e-8 * sqrt((double)d));
}

// deferred[j] = base + sel[j] (chunk-local query numbers -> batch-wide)
__global__ void defer_append_kernel(const int32_t* sel, int64_t n, int64_t base, int64_t* deferred) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j < n) deferred[j] = base + sel[j];
}

// out[rows[j], :] = sub[j, :] for the k-wide result rows of the deferred queries
__global__ void scatter_rows_kernel(const int64_t* rows, int64_t n, int k, const float* sub_sc, const int64_t* sub_id, float* out_sc,
                                    int64_t* out_id) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n * k) return;
    const int64_t j = t / k, o = t - j * k;
    out_sc[rows[j] * k + o] = sub_sc[t];
    out_id[rows[j] * k + o] = sub_id[t];
}

__global__ void fill_pad_kernel(float* sc, int64_t* id, int64_t total, float pad) {
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        sc[t] = pad;
        id[t] = -1;
    }
}

// level 0: the caller's search. For an fp32 store with a bf16 copy (X.filt16) and a small k it is the FIRST level of a two-level
// search: bf16 filter with a longer candidate list, the queries whose certificate fails are deferred, gathered and answered by
// a level-1 call (tf32 filter on the same store, then the dense path for what still fails) and scattered back.
int search_core(b2_index* idx, const MatView& X_in, int metric, const void* q_dev, int q_dtype, int64_t nq, int k,
                       const int64_t* id_map, int64_t id_offset, float* out_sc, int64_t* out_id, cudaStream_t st, int level) {
    if (level == 0) idx->last_filter_ms = -1.f;
    if (nq <= 0) return B2_OK;
    if (level == 0) g_stats[ST_QUERIES] += nq;
    // candidate capacity of the bf16 first level (the 2^-8 operand error lets more rows straddle the k-th score): 0 = not used
    const int kp16 = (X_in.filt16 && level == 0 && X_in.n >= 4096) ? (k <= 4 ? 32 : k <= 12 ? 64 : k <= 24 ? 96 : 0) : 0;
    MatView X = X_in;
    if (kp16) {
        X.filt = X_in.filt16;
        X.filt_pitch = X_in.filt16_pitch;
        X.filt_dtype = B2_BF16;
    }
    const bool defer = kp16 != 0;
    int64_t n_deferred = 0;
    if (X.n <= 0) {
        fill_pad_kernel<<<148, 256, 0, st>>>(out_sc, out_id, nq * k, metric == B2_METRIC_L2 ? FLT_MAX : -FLT_MAX);
        B2_LAUNCH_CHECK();
        return B2_OK;
    }
    const int kp = kp16 ? kp16 : filter_kp_for_k(k);
    const int min_splits = filter_min_splits_for_k(k);
    // the filter needs a corpus worth tiling: two tiles at least, and for k > 64 enough tiles to cut into min_splits splits
    // with k well below the rows of a split
    const bool use_filter = kp != 0 && X.n >= 512 && ceil_div(X.n, 256) >= min_splits && X.n >= 4 * (int64_t)k;
    const bool full_sort = k > dense_select_max_k();  // dense path sorts whole rows: score + two key buffers per column
    const int64_t dense_rows_cap = std::max<int64_t>(1, (int64_t)(512ull << 20) / (std::max<int64_t>(X.n, 1) * (full_sort ? 24 : 4)));
    if (!use_filter) {
        if (k > dense_max_k()) {
            set_error("k=%d is not supported (max %d)", k, dense_max_k());
            return B2_ERANGE;
        }
        const int64_t rows = std::min<int64_t>(dense_rows_cap, nq);
        B2_TRY(idx->dense.ensure((size_t)rows * X.n * sizeof(float)));
        if (full_sort) B2_TRY(idx->sort_keys.ensure(dense_sort_ws_bytes(rows, X.n)));
        B2_TRY(launch_dense_topk(X, q_dev, q_dtype, nq, nullptr, nq, metric, k, id_map, id_offset, idx->dense.as<float>(), rows,
                                 full_sort ? idx->sort_keys.as<uint64_t>() : nullptr, out_sc, out_id, st));
        g_stats[ST_FALLBACK] += nq;
        return B2_OK;
    }
    int dev_sms = 148;
    cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, idx->device);
    const int filt_dtype = X.filt_dtype;
    const int64_t q_pitch = round_up(X.d, filt_dtype == B2_F32 ? 4 : 8);
    const float rel_eps = filter_rel_eps(X.dtype, filt_dtype, q_dtype, X.d);
    // queries that already have the filter's element type and a TMA-compatible pitch are streamed in place
    const bool q_in_place = q_dtype == filt_dtype && q_pitch == X.d && (reinterpret_cast<uintptr_t>(q_dev) & 15) == 0;
    // bound the candidate workspace: process the queries in chunks
    // bound the candidate workspace (nqc x n_splits x kp x 8 bytes) to a few GB: fewer queries per chunk when k needs many splits
    const int64_t chunk = std::max<int64_t>(4096, std::min<int64_t>(1 << 20, (4LL << 30) / ((int64_t)std::max(min_splits, 8) * kp * 8)));
    for (int64_t q0 = 0; q0 < nq; q0 += chunk) {
        const int64_t nqc = std::min<int64_t>(chunk, nq - q0);
        const char* qc = reinterpret_cast<const char*>(q_dev) + (size_t)q0 * X.d * esize(q_dtype);
        float* osc = out_sc + (size_t)q0 * k;
        int64_t* oid = out_id + (size_t)q0 * k;
        const bool two_cta = filter_use_pair(nqc);
        int units_whole = 0;
        const int n_splits = filter_choose_splits(nqc, X.n, dev_sms, two_cta, false, min_splits, &units_whole);
        if (n_splits <= 0) {
            set_error("internal: no valid corpus split for k=%d over %lld rows", k, (long long)X.n);
            return B2_EINVAL;
        }
        if (!q_in_place) B2_TRY(idx->q_filt.ensure((size_t)nqc * q_pitch * esize(filt_dtype)));
        const void* q_filt = q_in_place ? static_cast<const void*>(qc) : idx->q_filt.p;
        B2_TRY(idx->cand_score.ensure((size_t)nqc * n_splits * kp * sizeof(float)));
        B2_TRY(idx->cand_id.ensure((size_t)nqc * n_splits * kp * sizeof(int32_t)));
        B2_TRY(idx->cand_thr.ensure((size_t)nqc * n_splits * 2 * sizeof(float)));  // two epilogue sets per split
        B2_TRY(idx->flags.ensure((size_t)nqc * sizeof(int32_t)));
        B2_TRY(idx->sel.ensure((size_t)(nqc + 1) * sizeof(int32_t)));  // [0] = counter, [1..] = uncertified queries
        B2_TRY(idx->h_flags.ensure(64));
        int32_t* sel_count = idx->sel.as<int32_t>();
        int32_t* sel_list = sel_count + 1;
        B2_CUDA(cudaMemsetAsync(sel_count, 0, sizeof(int32_t), st));
        // fp16 filter operands: queries with an element beyond fp16's finite range are flagged here and answered exactly
        int32_t* q_bad = nullptr;
        if (!q_in_place && filt_dtype == B2_F16) {
            B2_TRY(idx->q_bad.ensure((size_t)nqc * sizeof(int32_t)));
            q_bad = idx->q_bad.as<int32_t>();
            B2_CUDA(cudaMemsetAsync(q_bad, 0, (size_t)nqc * sizeof(int32_t), st));
        }
        if (!q_in_place) B2_TRY(launch_prep_queries(qc, q_dtype, nqc, X.d, idx->q_filt.p, filt_dtype, q_pitch, st, q_bad));
        B2_CUDA(cudaEventRecord(idx->ev0, st));
        B2_TRY(launch_knn_filter(X, q_filt, q_pitch, nqc, metric, kp, n_splits, two_cta, idx->cand_score.as<float>(),
                                 idx->cand_id.as<int32_t>(), idx->cand_thr.as<float>(), idx->device, st, false, units_whole));
        B2_CUDA(cudaEventRecord(idx->ev1, st));
        B2_TRY(launch_finalize(X, qc, q_dtype, nqc, metric, k, kp, kp / 2, 2 * n_splits, idx->cand_score.as<float>(),
                               idx->cand_id.as<int32_t>(), idx->cand_thr.as<float>(), rel_eps, id_map, id_offset, osc, oid,
                               idx->flags.as<int32_t>(), sel_list, sel_count, st, nullptr, q_bad));
        // the certificate outcome comes back as ONE counter (the failed queries are compacted on the device)
        int32_t* h_count = reinterpret_cast<int32_t*>(idx->h_flags.p);
        B2_CUDA(cudaMemcpyAsync(h_count, sel_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        cudaError_t se = cudaStreamSynchronize(st);
        if (se != cudaSuccess) {
            set_error("search pipeline failed on the device: %s", cudaGetErrorString(se));
            return B2_ECUDA;
        }
        float ms = -1.f;
        if (cudaEventElapsedTime(&ms, idx->ev0, idx->ev1) == cudaSuccess)
            idx->last_filter_ms = (idx->last_filter_ms < 0 ? 0.f : idx->last_filter_ms) + ms;
        // exact fallback for the queries the certificate could not cover
        const int64_t n_sel = *h_count;
        if (n_sel > 0 && defer) {
            B2_TRY(idx->defer.ensure((size_t)nq * sizeof(int64_t)));
            defer_append_kernel<<<(unsigned)ceil_div(n_sel, 256), 256, 0, st>>>(sel_list, n_sel, q0, idx->defer.as<int64_t>() + n_deferred);
            B2_LAUNCH_CHECK();
            n_deferred += n_sel;
        } else if (n_sel > 0) {
            if (k > dense_max_k()) {
                set_error("internal: fallback with k=%d", k);
                return B2_ERANGE;
            }
            g_stats[ST_FALLBACK] += n_sel;
            const int64_t rows = std::min<int64_t>(dense_rows_cap, n_sel);
            B2_TRY(idx->dense.ensure((size_t)rows * X.n * sizeof(float)));
            B2_TRY(launch_dense_topk(X, qc, q_dtype, nqc, sel_list, n_sel, metric, k, id_map, id_offset, idx->dense.as<float>(), rows,
                                     nullptr, osc, oid, st));
        }
    }
    if (n_deferred > 0) {
        // second level: the deferred queries against the exact-operand (tf32) filter of the same store
        const size_t qrow = (size_t)X.d * esize(q_dtype);
        B2_TRY(idx->q_sub.ensure((size_t)n_deferred * qrow));
        B2_TRY(idx->sub_sc.ensure((size_t)n_deferred * k * sizeof(float)));
        B2_TRY(idx->sub_id.ensure((size_t)n_deferred * k * sizeof(int64_t)));
        B2_TRY(idx->scalar.ensure(64));
        int* err = reinterpret_cast<int*>(idx->scalar.as<char>() + 16);
        B2_TRY(launch_gather_rows(q_dev, q_dtype, X.d, idx->defer.as<int64_t>(), n_deferred, nq, idx->q_sub.p, err, st));
        MatView X2 = X_in;
        X2.filt16 = nullptr;
        B2_TRY(search_core(idx, X2, metric, idx->q_sub.p, q_dtype, n_deferred, k, id_map, id_offset, idx->sub_sc.as<float>(),
                           idx->sub_id.as<int64_t>(), st, /*level=*/1));
        scatter_rows_kernel<<<(unsigned)ceil_div(n_deferred * k, 256), 256, 0, st>>>(idx->defer.as<int64_t>(), n_deferred, k, idx->sub_sc.as<float>(),
                                                                                    idx->sub_id.as<int64_t>(), out_sc, out_id);
        B2_LAUNCH_CHECK();
        g_stats[ST_SECOND_LEVEL] += n_deferred;
    }
    return B2_OK;
}

// searchable view for an ids subset (faiss_vs.py:57-64: temporary index over vecs[ids])
static int build_subset(b2_index* idx, const int64_t* ids_dev, int64_t m, MatView& sub, cudaStream_t st) {
    B2_TRY(idx->sub_store.ensure((size_t)std::max<int64_t>(m, 1) * idx->d * esize(idx->dtype)));
    B2_TRY(idx->scalar.ensure(64));
    int* err = reinterpret_cast<int*>(idx->scalar.as<char>() + 16);
    B2_CUDA(cudaMemsetAsync(err, 0, sizeof(int), st));
    B2_TRY(launch_gather_rows(idx->store.p, idx->dtype, idx->d, ids_dev, m, idx->n, idx->sub_store.p, err, st));
    int herr = 0;
    B2_CUDA(cudaMemcpyAsync(&herr, err, sizeof(int), cudaMemcpyDeviceToHost, st));
    B2_CUDA(cudaStreamSynchronize(st));
    if (herr) {
        set_error("ids contains a position outside [0, %lld)", (long long)idx->n);
        return B2_ERANGE;
    }
    return build_view(idx->sub_store.p, m, idx->d, idx->dtype, idx->sub_filt, idx->sub_norm2, idx->scalar, sub, st, &idx->sub_filt16);
}

}  // namespace b2

// =====================================================================================================================
extern "C" {

int b2_abi_version(void) { return B2_ABI_VERSION; }
const char* b2_last_error(void) { return g_err.c_str(); }

int b2_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    int ok = 0;
    for (int i = 0; i < n; ++i) {
        int major = 0;
        cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i);
        if (major == 10) ok++;
    }
    return ok;
}

int b2_max_k(void) { return dense_max_k(); }

int b2_index_create(const void* x, int64_t n, int32_t d, int32_t dtype, int32_t metric, int32_t device, int32_t x_on_device,
                    b2_index** out) {
    if (!out) { set_error("out is NULL"); return B2_EINVAL; }
    *out = nullptr;
    if (n < 0 || d <= 0 || (n > 0 && !x)) { set_error("bad matrix shape n=%lld d=%d", (long long)n, d); return B2_EINVAL; }
    if (dtype != B2_F32 && dtype != B2_BF16 && dtype != B2_F16) { set_error("dtype must be B2_F32, B2_BF16 or B2_F16"); return B2_EINVAL; }
    if (metric != B2_METRIC_IP && metric != B2_METRIC_L2) { set_error("metric must be B2_METRIC_IP or B2_METRIC_L2"); return B2_EINVAL; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device: libb2lotus has no CPU fallback");
        return B2_ENODEV;
    }
    if (device < 0 || device >= ndev) { set_error("device %d out of range (%d visible)", device, ndev); return B2_EINVAL; }
    int major = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
    if (major != 10) { set_error("device %d is sm_%d0; this library is built for sm_100a (B200) only", device, major); return B2_ENODEV; }
    DeviceGuard guard(device);
    b2_index* idx = new b2_index();
    idx->device = device;
    idx->n = n;
    idx->d = d;
    idx->dtype = dtype;
    idx->metric = metric;
    auto fail = [&](int rc) { b2_index_free(idx); return rc; };
    if (cudaStreamCreateWithFlags(&idx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&idx->ev0) != cudaSuccess || cudaEventCreate(&idx->ev1) != cudaSuccess) {
        set_error("stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
        return fail(B2_ECUDA);
    }
    const size_t bytes = (size_t)std::max<int64_t>(n, 1) * d * esize(dtype);
    int rc = idx->store.ensure(bytes);
    if (rc != B2_OK) return fail(rc);
    if (n > 0) {
        // a device-resident source was produced on some other stream (e.g. torch's): our private stream is
        // non-blocking, so order the copy after everything already submitted to the device
        if (x_on_device && cudaDeviceSynchronize() != cudaSuccess) {
            set_error("device synchronisation before the copy failed: %s", cudaGetErrorString(cudaGetLastError()));
            return fail(B2_ECUDA);
        }
        cudaError_t e = cudaMemcpyAsync(idx->store.p, x, (size_t)n * d * esize(dtype),
                                        x_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, idx->stream);
        if (e != cudaSuccess) { set_error("copy of the matrix failed: %s", cudaGetErrorString(e)); return fail(B2_ECUDA); }
    }
    rc = build_view(idx->store.p, n, d, dtype, idx->filt_pad, idx->norm2, idx->scalar, idx->view, idx->stream, &idx->filt16);
    if (rc != B2_OK) return fail(rc);
    *out = idx;
    return B2_OK;
}

void b2_index_free(b2_index* idx) {
    if (!idx) return;
    DeviceGuard guard(idx->device);
    DevBuf* bufs[] = {&idx->store, &idx->filt_pad, &idx->filt16, &idx->sub_filt16, &idx->defer, &idx->q_sub, &idx->sub_sc, &idx->sub_id, &idx->q_norm2, &idx->q_bad, &idx->norm2, &idx->scalar, &idx->q_in, &idx->q_filt, &idx->cand_score,
                      &idx->cand_id, &idx->cand_thr, &idx->flags, &idx->sel, &idx->dense, &idx->out_sc, &idx->out_id,
                      &idx->ids_dev, &idx->sub_store, &idx->sub_filt, &idx->sub_norm2, &idx->sort_keys};
    for (DevBuf* b : bufs) b->release();
    idx->h_flags.release();
    km_work_free(idx->km);
    idx->km = nullptr;
    if (idx->ev0) cudaEventDestroy(idx->ev0);
    if (idx->ev1) cudaEventDestroy(idx->ev1);
    if (idx->stream) cudaStreamDestroy(idx->stream);
    delete idx;
}

int64_t b2_index_ntotal(const b2_index* idx) { return idx ? idx->n : -1; }
int32_t b2_index_dim(const b2_index* idx) { return idx ? idx->d : -1; }
int32_t b2_index_dtype(const b2_index* idx) { return idx ? idx->dtype : -1; }
int32_t b2_index_metric(const b2_index* idx) { return idx ? idx->metric : -1; }
int32_t b2_index_device(const b2_index* idx) { return idx ? idx->device : -1; }
const void* b2_index_data_dev(const b2_index* idx) { return idx ? idx->store.p : nullptr; }
float b2_last_filter_ms(const b2_index* idx) { return idx ? idx->last_filter_ms : -1.f; }

static int check_search_args(b2_index* idx, const void* q, int64_t nq, int32_t q_dtype, int32_t k) {
    if (!idx) { set_error("Index not loaded"); return B2_EINVAL; }
    if (nq < 0 || (nq > 0 && !q)) { set_error("bad query batch"); return B2_EINVAL; }
    if (q_dtype != B2_F32 && q_dtype != B2_BF16 && q_dtype != B2_F16) { set_error("q_dtype must be B2_F32, B2_BF16 or B2_F16"); return B2_EINVAL; }
    if (k <= 0) { set_error("k must be positive (got %d)", k); return B2_EINVAL; }
    if (k > dense_max_k()) { set_error("k=%d is not supported (max %d)", k, dense_max_k()); return B2_ERANGE; }
    return B2_OK;
}

int b2_index_search_dev(b2_index* idx, const void* q_dev, int64_t nq, int32_t q_dtype, int32_t k, const int64_t* ids_dev,
                        int64_t n_ids, int64_t id_offset, float* out_scores_dev, int64_t* out_idx_dev, void* stream) {
    B2_TRY(check_search_args(idx, q_dev, nq, q_dtype, k));
    if (nq == 0) return B2_OK;
    if (!out_scores_dev || !out_idx_dev) { set_error("output buffers are NULL"); return B2_EINVAL; }
    DeviceGuard guard(idx->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (ids_dev) {
        if (n_ids < 0) { set_error("n_ids < 0"); return B2_EINVAL; }
        MatView sub;
        B2_TRY(build_subset(idx, ids_dev, n_ids, sub, st));
        B2_TRY(search_core(idx, sub, idx->metric, q_dev, q_dtype, nq, k, ids_dev, 0, out_scores_dev, out_idx_dev, st));
    } else {
        B2_TRY(search_core(idx, idx->view, idx->metric, q_dev, q_dtype, nq, k, nullptr, id_offset, out_scores_dev, out_idx_dev, st));
    }
    B2_CUDA(cudaStreamSynchronize(st));
    return B2_OK;
}

int b2_index_search(b2_index* idx, const void* q, int64_t nq, int32_t q_dtype, int32_t k, const int64_t* ids, int64_t n_ids,
                    float* out_scores, int64_t* out_idx) {
    B2_TRY(check_search_args(idx, q, nq, q_dtype, k));
    if (nq == 0) return B2_OK;
    if (!out_scores || !out_idx) { set_error("output buffers are NULL"); return B2_EINVAL; }
    DeviceGuard guard(idx->device);
    cudaStream_t st = idx->stream;
    const size_t qbytes = (size_t)nq * idx->d * esize(q_dtype);
    B2_TRY(idx->q_in.ensure(qbytes));
    B2_TRY(idx->out_sc.ensure((size_t)nq * k * sizeof(float)));
    B2_TRY(idx->out_id.ensure((size_t)nq * k * sizeof(int64_t)));
    B2_CUDA(cudaMemcpyAsync(idx->q_in.p, q, qbytes, cudaMemcpyHostToDevice, st));
    const int64_t* ids_dev = nullptr;
    if (ids) {
        if (n_ids < 0) { set_error("n_ids < 0"); return B2_EINVAL; }
        bool identity = n_ids == idx->n;
        for (int64_t i = 0; identity && i < n_ids; ++i) identity = ids[i] == i;
        if (!identity) {
            B2_TRY(idx->ids_dev.ensure((size_t)std::max<int64_t>(n_ids, 1) * sizeof(int64_t)));
            B2_CUDA(cudaMemcpyAsync(idx->ids_dev.p, ids, (size_t)n_ids * sizeof(int64_t), cudaMemcpyHostToDevice, st));
            ids_dev = idx->ids_dev.as<int64_t>();
        }
    }
    if (ids_dev) {
        MatView sub;
        B2_TRY(build_subset(idx, ids_dev, n_ids, sub, st));
        B2_TRY(search_core(idx, sub, idx->metric, idx->q_in.p, q_dtype, nq, k, ids_dev, 0, idx->out_sc.as<float>(), idx->out_id.as<int64_t>(), st));
    } else {
        B2_TRY(search_core(idx, idx->view, idx->metric, idx->q_in.p, q_dtype, nq, k, nullptr, 0, idx->out_sc.as<float>(),
                           idx->out_id.as<int64_t>(), st));
    }
    B2_CUDA(cudaMemcpyAsync(out_scores, idx->out_sc.p, (size_t)nq * k * sizeof(float), cudaMemcpyDeviceToHost, st));
    B2_CUDA(cudaMemcpyAsync(out_idx, idx->out_id.p, (size_t)nq * k * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { set_error("search failed on the device: %s", cudaGetErrorString(e)); return B2_ECUDA; }
    return B2_OK;
}

int b2_merge_topk_dev(const float* scores_dev, const int64_t* idx_dev, int32_t g, int64_t nq, int32_t k, int32_t metric,
                      int32_t device, float* out_scores_dev, int64_t* out_idx_dev, void* stream) {
    if (g <= 0 || k <= 0 || nq < 0) { set_error("bad merge shape g=%d nq=%lld k=%d", g, (long long)nq, k); return B2_EINVAL; }
    if (nq == 0) return B2_OK;
    if (!scores_dev || !idx_dev || !out_scores_dev || !out_idx_dev) { set_error("NULL buffer"); return B2_EINVAL; }
    DeviceGuard guard(device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    B2_TRY(launch_merge_topk(scores_dev, idx_dev, g, nq, k, metric, out_scores_dev, out_idx_dev, st));
    B2_CUDA(cudaStreamSynchronize(st));
    return B2_OK;
}

int b2_index_search_packed_dev(b2_index* idx, const void* q_dev, int64_t nq, int32_t q_dtype, int32_t k, uint64_t* out_packed_dev,
                               void* stream) {
    B2_TRY(check_search_args(idx, q_dev, nq, q_dtype, k));
    if (nq == 0) return B2_OK;
    if (!out_packed_dev) { set_error("output buffer is NULL"); return B2_EINVAL; }
    if (idx->n > 0xfffffffeLL) { set_error("packed lists hold 32-bit local ids"); return B2_ERANGE; }
    DeviceGuard guard(idx->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    B2_TRY(idx->out_sc.ensure((size_t)nq * k * sizeof(float)));
    B2_TRY(idx->out_id.ensure((size_t)nq * k * sizeof(int64_t)));
    B2_TRY(search_core(idx, idx->view, idx->metric, q_dev, q_dtype, nq, k, nullptr, 0, idx->out_sc.as<float>(), idx->out_id.as<int64_t>(), st));
    B2_TRY(launch_pack_topk(idx->out_sc.as<float>(), idx->out_id.as<int64_t>(), nq * (int64_t)k, out_packed_dev, st));
    B2_CUDA(cudaStreamSynchronize(st));
    return B2_OK;
}

// ---- row-sharded search in two stages ---------------------------------------------------------------------------------------
// stage 1: filter this shard, report per query a lower bound on the exact score of its j best local candidates (asynchronous:
// nothing is copied to the host). The caller all-reduces (MIN) the bounds over the ranks with j = ceil(k / ranks): k rows of the
// whole index are then known to reach that score. stage 2: finalize with that bound as a hint — rows that cannot reach it are
// not re-scored and the certificate only has to beat the hint — and pack. Shapes the staged path does not cover (dense path,
// fp32 two-level search, more than one query chunk, too many candidate entries) report -inf bounds and stage 2 runs the plain
// search, so the pair of calls is always valid.
int b2_index_search_stage1_dev(b2_index* idx, const void* q_dev, int64_t nq, int32_t q_dtype, int32_t k, int32_t j, float* lower_dev,
                               void* stream) {
    B2_TRY(check_search_args(idx, q_dev, nq, q_dtype, k));
    if (nq == 0) return B2_OK;
    if (!lower_dev || j <= 0) { set_error("bad stage-1 arguments"); return B2_EINVAL; }
    DeviceGuard guard(idx->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    b2_index::Staged& sg = idx->staged;
    sg = b2_index::Staged();
    sg.active = true;
    sg.q = q_dev;
    sg.nq = nq;
    sg.q_dtype = q_dtype;
    sg.k = k;
    const MatView& X = idx->view;
    const int kp = filter_kp_for_k(k);
    const int min_splits = filter_min_splits_for_k(k);
    const bool use_filter = kp != 0 && X.n >= 512 && ceil_div(X.n, 256) >= min_splits && X.n >= 4 * (int64_t)k;
    const bool two_level = X.filt16 != nullptr && k <= 24 && X.n >= 4096;
    const int64_t chunk = std::max<int64_t>(4096, std::min<int64_t>(1 << 20, (4LL << 30) / ((int64_t)std::max(min_splits, 8) * kp * 8)));
    int dev_sms = 148;
    cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, idx->device);
    const bool two_cta = filter_use_pair(nq);
    int units_whole = 0;
    const int n_splits = use_filter ? filter_choose_splits(nq, X.n, dev_sms, two_cta, false, min_splits, &units_whole) : 0;
    if (!use_filter || two_level || nq > chunk || n_splits <= 0 || 2 * n_splits * (kp / 2) > shard_lower_bound_max_entries() || j > k) {
        return launch_fill_f32(lower_dev, nq, -INFINITY, st);  // stage 2 will run the plain search
    }
    idx->last_filter_ms = -1.f;
    const int filt_dtype = X.filt_dtype;
    const int64_t q_pitch = round_up(X.d, filt_dtype == B2_F32 ? 4 : 8);
    const bool q_in_place = q_dtype == filt_dtype && q_pitch == X.d && (reinterpret_cast<uintptr_t>(q_dev) & 15) == 0;
    sg.q_bad = !q_in_place && filt_dtype == B2_F16;
    if (sg.q_bad) {
        B2_TRY(idx->q_bad.ensure((size_t)nq * sizeof(int32_t)));
        B2_CUDA(cudaMemsetAsync(idx->q_bad.p, 0, (size_t)nq * sizeof(int32_t), st));
    }
    if (!q_in_place) {
        B2_TRY(idx->q_filt.ensure((size_t)nq * q_pitch * esize(filt_dtype)));
        B2_TRY(launch_prep_queries(q_dev, q_dtype, nq, X.d, idx->q_filt.p, filt_dtype, q_pitch, st,
                                   sg.q_bad ? idx->q_bad.as<int32_t>() : nullptr));
    }
    const void* q_filt = q_in_place ? q_dev : idx->q_filt.p;
    B2_TRY(idx->cand_score.ensure((size_t)nq * n_splits * kp * sizeof(float)));
    B2_TRY(idx->cand_id.ensure((size_t)nq * n_splits * kp * sizeof(int32_t)));
    B2_TRY(idx->cand_thr.ensure((size_t)nq * n_splits * 2 * sizeof(float)));
    B2_TRY(idx->q_norm2.ensure((size_t)nq * sizeof(float)));
    B2_TRY(idx->scalar.ensure(64));
    B2_CUDA(cudaEventRecord(idx->ev0, st));
    B2_TRY(launch_knn_filter(X, q_filt, q_pitch, nq, idx->metric, kp, n_splits, two_cta, idx->cand_score.as<float>(), idx->cand_id.as<int32_t>(),
                             idx->cand_thr.as<float>(), idx->device, st, false, units_whole));
    B2_CUDA(cudaEventRecord(idx->ev1, st));
    sg.kp = kp;
    sg.n_splits = n_splits;
    sg.rel_eps = filter_rel_eps(X.dtype, filt_dtype, q_dtype, X.d);
    sg.abs_eps = filter_abs_eps(X.dtype, filt_dtype, q_dtype, X.d);
    sg.filtered = true;
    B2_TRY(launch_row_norms(q_dev, q_dtype, nq, X.d, idx->q_norm2.as<float>(), idx->scalar.as<float>() + 8, st));
    B2_TRY(launch_shard_lower_bound(idx->cand_score.as<float>(), idx->cand_id.as<int32_t>(), nq, 2 * n_splits, kp / 2, j, idx->q_norm2.as<float>(),
                                    X.max_norm, sg.rel_eps, sg.abs_eps, sg.q_bad ? idx->q_bad.as<int32_t>() : nullptr, idx->metric,
                                    lower_dev, st));
    g_stats[ST_QUERIES] += nq;
    return B2_OK;
}

int b2_index_search_stage2_packed_dev(b2_index* idx, const float* hint_dev, uint64_t* out_packed_dev, void* stream) {
    if (!idx) { set_error("Index not loaded"); return B2_EINVAL; }
    b2_index::Staged sg = idx->staged;
    idx->staged.active = false;
    if (!sg.active) { set_error("stage 2 without a stage 1"); return B2_EINVAL; }
    if (!out_packed_dev) { set_error("output buffer is NULL"); return B2_EINVAL; }
    if (!sg.filtered) return b2_index_search_packed_dev(idx, sg.q, sg.nq, sg.q_dtype, sg.k, out_packed_dev, stream);
    if (idx->n > 0xfffffffeLL) { set_error("packed lists hold 32-bit local ids"); return B2_ERANGE; }
    DeviceGuard guard(idx->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const MatView& X = idx->view;
    const int64_t nq = sg.nq;
    const int k = sg.k;
    B2_TRY(idx->out_sc.ensure((size_t)nq * k * sizeof(float)));
    B2_TRY(idx->out_id.ensure((size_t)nq * k * sizeof(int64_t)));
    B2_TRY(idx->flags.ensure((size_t)nq * sizeof(int32_t)));
    B2_TRY(idx->sel.ensure((size_t)(nq + 1) * sizeof(int32_t)));
    B2_TRY(idx->h_flags.ensure(64));
    int32_t* sel_count = idx->sel.as<int32_t>();
    int32_t* sel_list = sel_count + 1;
    B2_CUDA(cudaMemsetAsync(sel_count, 0, sizeof(int32_t), st));
    B2_TRY(launch_finalize(X, sg.q, sg.q_dtype, nq, idx->metric, k, sg.kp, sg.kp / 2, 2 * sg.n_splits, idx->cand_score.as<float>(),
                           idx->cand_id.as<int32_t>(), idx->cand_thr.as<float>(), sg.rel_eps, nullptr, 0, idx->out_sc.as<float>(),
                           idx->out_id.as<int64_t>(), idx->flags.as<int32_t>(), sel_list, sel_count, st, hint_dev,
                           sg.q_bad ? idx->q_bad.as<int32_t>() : nullptr));
    int32_t* h_count = reinterpret_cast<int32_t*>(idx->h_flags.p);
    B2_CUDA(cudaMemcpyAsync(h_count, sel_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    cudaError_t se = cudaStreamSynchronize(st);
    if (se != cudaSuccess) { set_error("search pipeline failed on the device: %s", cudaGetErrorString(se)); return B2_ECUDA; }
    float ms = -1.f;
    if (cudaEventElapsedTime(&ms, idx->ev0, idx->ev1) == cudaSuccess) idx->last_filter_ms = ms;
    const int64_t n_sel = *h_count;
    if (n_sel > 0) {  // uncertified queries: the exact local top-k (a superset of what the merge needs)
        g_stats[ST_FALLBACK] += n_sel;
        const int64_t rows = std::min<int64_t>(std::max<int64_t>(1, (int64_t)(512ull << 20) / (std::max<int64_t>(X.n, 1) * 4)), n_sel);
        B2_TRY(idx->dense.ensure((size_t)rows * X.n * sizeof(float)));
        B2_TRY(launch_dense_topk(X, sg.q, sg.q_dtype, nq, sel_list, n_sel, idx->metric, k, nullptr, 0, idx->dense.as<float>(), rows, nullptr,
                                 idx->out_sc.as<float>(), idx->out_id.as<int64_t>(), st));
    }
    B2_TRY(launch_pack_topk(idx->out_sc.as<float>(), idx->out_id.as<int64_t>(), nq * (int64_t)k, out_packed_dev, st));
    B2_CUDA(cudaStreamSynchronize(st));
    return B2_OK;
}

int b2_merge_topk_packed_dev(const uint64_t* packed_dev, const int64_t* shard_offsets, int32_t g, int64_t nq, int32_t k, int32_t metric,
                             int32_t device, float* out_scores_dev, int64_t* out_idx_dev, void* stream) {
    if (g <= 0 || k <= 0 || nq < 0 || !shard_offsets) { set_error("bad merge shape g=%d nq=%lld k=%d", g, (long long)nq, k); return B2_EINVAL; }
    if (nq == 0) return B2_OK;
    if (!packed_dev || !out_scores_dev || !out_idx_dev) { set_error("NULL buffer"); return B2_EINVAL; }
    DeviceGuard guard(device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    B2_TRY(launch_merge_packed(packed_dev, shard_offsets, g, nq, k, metric, out_scores_dev, out_idx_dev, st));
    B2_CUDA(cudaStreamSynchronize(st));
    return B2_OK;
}

int b2_index_gather(b2_index* idx, const int64_t* ids, int64_t m, void* out, int32_t out_on_device) {
    if (!idx) { set_error("Index not loaded"); return B2_EINVAL; }
    if (m < 0 || (m > 0 && (!ids || !out))) { set_error("bad gather arguments"); return B2_EINVAL; }
    if (m == 0) return B2_OK;
    DeviceGuard guard(idx->device);
    cudaStream_t st = idx->stream;
    const size_t row_bytes = (size_t)idx->d * esize(idx->dtype);
    B2_TRY(idx->scalar.ensure(64));
    int* err = reinterpret_cast<int*>(idx->scalar.as<char>() + 16);
    B2_CUDA(cudaMemsetAsync(err, 0, sizeof(int), st));
    const int64_t* ids_dev = ids;
    void* out_dev = out;
    if (!out_on_device) {
        B2_TRY(idx->ids_dev.ensure((size_t)m * sizeof(int64_t)));
        B2_CUDA(cudaMemcpyAsync(idx->ids_dev.p, ids, (size_t)m * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        ids_dev = idx->ids_dev.as<int64_t>();
        B2_TRY(idx->sub_store.ensure((size_t)m * row_bytes));
        out_dev = idx->sub_store.p;
    }
    B2_TRY(launch_gather_rows(idx->store.p, idx->dtype, idx->d, ids_dev, m, idx->n, out_dev, err, st));
    int herr = 0;
    B2_CUDA(cudaMemcpyAsync(&herr, err, sizeof(int), cudaMemcpyDeviceToHost, st));
    if (!out_on_device) B2_CUDA(cudaMemcpyAsync(out, out_dev, (size_t)m * row_bytes, cudaMemcpyDeviceToHost, st));
    B2_CUDA(cudaStreamSynchronize(st));
    if (herr) { set_error("ids contains a position outside [0, %lld)", (long long)idx->n); return B2_ERANGE; }
    return B2_OK;
}

// Host-side marshalling helper (no device work): round-to-nearest-even fp32 -> bf16 bit patterns, NaN kept quiet, and
// report whether every value was already bf16-representable (then the 2-byte form is EXACT and the plugin ships it).
int b2_host_f32_to_bf16(const float* x, int64_t count, uint16_t* out, int32_t* all_exact) {
    if (count < 0 || (count > 0 && (!x || !out))) { set_error("bad conversion arguments"); return B2_EINVAL; }
    const int64_t kChunk = 1 << 20;
    const int64_t nchunks = (count + kChunk - 1) / kChunk;
    unsigned hw = std::thread::hardware_concurrency();
    const int nthreads = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(hw ? hw : 1, 16), nchunks));
    std::atomic<int64_t> next{0};
    std::atomic<int> inexact{0};
    auto work = [&]() {
        int local_inexact = 0;
        for (;;) {
            const int64_t c = next.fetch_add(1);
            if (c >= nchunks) break;
            const int64_t lo = c * kChunk, hi = std::min(count, lo + kChunk);
            const uint32_t* u = reinterpret_cast<const uint32_t*>(x);
            for (int64_t i = lo; i < hi; ++i) {
                const uint32_t v = u[i];
                local_inexact |= (v & 0xffffu) != 0;
                const bool is_nan = (v & 0x7fffffffu) > 0x7f800000u;
                out[i] = is_nan ? (uint16_t)((v >> 16) | 0x0040u) : (uint16_t)((v + 0x7fffu + ((v >> 16) & 1u)) >> 16);
            }
        }
        if (local_inexact) inexact.store(1);
    };
    if (nthreads <= 1) {
        work();
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < nthreads; ++t) pool.emplace_back(work);
        for (auto& t : pool) t.join();
    }
    if (all_exact) *all_exact = inexact.load() ? 0 : 1;
    return B2_OK;
}

// Host-side marshalling helper: bf16 bit patterns -> float32 (exact), threaded.
int b2_host_bf16_to_f32(const uint16_t* x, int64_t count, float* out) {
    if (count < 0 || (count > 0 && (!x || !out))) { set_error("bad conversion arguments"); return B2_EINVAL; }
    const int64_t kChunk = 1 << 20;
    const int64_t nchunks = (count + kChunk - 1) / kChunk;
    unsigned hw = std::thread::hardware_concurrency();
    const int nthreads = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(hw ? hw : 1, 16), nchunks));
    std::atomic<int64_t> next{0};
    auto work = [&]() {
        uint32_t* o = reinterpret_cast<uint32_t*>(out);
        for (;;) {
            const int64_t c = next.fetch_add(1);
            if (c >= nchunks) break;
            const int64_t lo = c * kChunk, hi = std::min(count, lo + kChunk);
            for (int64_t i = lo; i < hi; ++i) o[i] = (uint32_t)x[i] << 16;
        }
    };
    if (nthreads <= 1) {
        work();
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < nthreads; ++t) pool.emplace_back(work);
        for (auto& t : pool) t.join();
    }
    return B2_OK;
}

// The filter's work schedule for a (queries, rows, k) shape on `num_sms` SMs — no device work: lets the CPU test-suite check that
// every (query unit, corpus tile) pair is covered exactly once for the shapes the GPU tests do not reach.
int b2_debug_filter_plan(int64_t nq, int64_t n, int32_t k, int32_t num_sms, int32_t* kp, int32_t* n_splits, int32_t* units_whole,
                         int32_t* two_cta) {
    if (nq <= 0 || n <= 0 || k <= 0 || num_sms <= 0 || !kp || !n_splits || !units_whole || !two_cta) { set_error("bad arguments"); return B2_EINVAL; }
    *kp = filter_kp_for_k(k);
    *two_cta = filter_use_pair(nq) ? 1 : 0;
    int uw = 0;
    *n_splits = *kp ? filter_choose_splits(nq, n, num_sms, *two_cta != 0, false, filter_min_splits_for_k(k), &uw) : 0;
    *units_whole = uw;
    return B2_OK;
}

int b2_stats(int64_t* out, int32_t cap) {
    int n = cap < 8 ? cap : 8;
    for (int i = 0; i < n; ++i) out[i] = g_stats[i];
    return n;
}
void b2_stats_reset(void) { memset(g_stats, 0, sizeof(g_stats)); }

}  // extern "C"
