// dedup.cu — sem_dedup's data-parallel core (lotus/sem_ops/sem_dedup.py:45-84) without the N x N DataFrame:
//   b2_threshold_pairs     : tcgen05 all-pairs filter (upper triangle only) -> exact canonical verification of the
//                            candidates with the reference's strict `score > threshold` -> pair list sorted by (i, j)
//   b2_connected_components: lock-free union-find (link larger root under smaller root) + path compression;
//                            label = smallest row id of the component, the deterministic stand-in for the
//                            reference's DFS over a Python set (sem_dedup.py:58-82)
#include <algorithm>
#include <vector>

#include "index.cuh"

namespace b2 {
namespace {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ void load_group2(const char* row, int dtype, int g, int d, bool vec, float (&o)[4]) {
    const int i0 = g * 4;
    if (vec) {
        if (dtype == B2_F32) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(row) + g);
            o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
        } else if (dtype == B2_F16) {
            const uint2 t = __ldg(reinterpret_cast<const uint2*>(row) + g);
            const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&t.x));
            const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
            o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
        } else {
            const uint2 t = __ldg(reinterpret_cast<const uint2*>(row) + g);
            o[0] = __uint_as_float(t.x << 16);
            o[1] = __uint_as_float(t.x & 0xffff0000u);
            o[2] = __uint_as_float(t.y << 16);
            o[3] = __uint_as_float(t.y & 0xffff0000u);
        }
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int i = i0 + e;
            o[e] = i >= d             ? 0.f
                   : dtype == B2_F32 ? reinterpret_cast<const float*>(row)[i]
                   : dtype == B2_F16 ? __half2float(reinterpret_cast<const __half*>(row)[i])
                                     : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(row)[i]);
        }
    }
}

// one warp per candidate pair: canonical inner product (same order as oracle orc_dot_canonical), strict compare
__global__ void pair_verify_kernel(const char* store, int dtype, int d, const int32_t* ci, const int32_t* cj, int64_t ncand,
                                   float thr, int32_t* out_i, int32_t* out_j, unsigned long long* out_count) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const bool vec = (d % 4) == 0;
    const size_t row_bytes = (size_t)d * (dtype == B2_F32 ? 4 : 2);
    const int ngroups = (d + 3) >> 2;
    for (int64_t c = warp; c < ncand; c += nwarps) {
        const int i = ci[c], j = cj[c];
        const char* ri = store + (size_t)i * row_bytes;
        const char* rj = store + (size_t)j * row_bytes;
        double acc = 0.0;
        for (int g = lane; g < ngroups; g += 32) {
            float a[4], b[4];
            load_group2(ri, dtype, g, d, vec, a);
            load_group2(rj, dtype, g, d, vec, b);
#pragma unroll
            for (int e = 0; e < 4; ++e) acc = fma((double)a[e], (double)b[e], acc);
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(FULL, acc, off);
        if (lane == 0 && (float)acc > thr) {
            const unsigned long long pos = atomicAdd(out_count, 1ull);
            out_i[pos] = i;
            out_j[pos] = j;
        }
    }
}

// ---- union-find -----------------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t uf_find(int64_t* parent, int64_t a) {
    int64_t p = parent[a];
    while (p != a) {
        const int64_t gp = parent[p];
        if (gp != p) parent[a] = gp;  // path halving (benign race: parents only ever move towards the root)
        a = p;
        p = gp;
    }
    return a;
}

__global__ void uf_init_kernel(int64_t* parent, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) parent[i] = i;
}

__global__ void uf_union_kernel(int64_t* parent, const int64_t* pi, const int64_t* pj, int64_t m, int64_t n, int* err) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < m; e += (int64_t)gridDim.x * blockDim.x) {
        int64_t a = pi[e], b = pj[e];
        if (a < 0 || b < 0 || a >= n || b >= n) {
            atomicExch(err, 1);
            continue;
        }
        while (true) {
            a = uf_find(parent, a);
            b = uf_find(parent, b);
            if (a == b) break;
            if (a < b) { const int64_t t = a; a = b; b = t; }  // a = larger root, goes under b
            const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(parent + a),
                                                     (unsigned long long)a, (unsigned long long)b);
            if (old == (unsigned long long)a) break;  // linked; otherwise someone moved a: retry from the new roots
        }
    }
}

__global__ void uf_flatten_kernel(int64_t* parent, int64_t* labels, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t a = i;
        while (parent[a] != a) a = parent[a];
        labels[i] = a;  // roots only ever link to smaller ids: the root is the component's minimum
    }
}

}  // namespace
}  // namespace b2

using namespace b2;

extern "C" {

int b2_threshold_pairs(b2_index* idx, float threshold, int32_t part, int32_t nparts, int64_t* out_i, int64_t* out_j, int64_t cap,
                       int64_t* n_pairs) {
    if (!idx) { set_error("Index not loaded"); return B2_EINVAL; }
    if (!n_pairs || cap < 0 || (cap > 0 && (!out_i || !out_j))) { set_error("bad output buffers"); return B2_EINVAL; }
    if (nparts <= 0 || part < 0 || part >= nparts) { set_error("bad part/nparts %d/%d", part, nparts); return B2_EINVAL; }
    if (idx->metric != B2_METRIC_IP) { set_error("threshold_pairs is defined for inner-product indexes (sem_dedup thresholds a similarity)"); return B2_EINVAL; }
    *n_pairs = 0;
    if (idx->n < 2) return B2_OK;
    DeviceGuard guard(idx->device);
    cudaStream_t st = idx->stream;
    const MatView& X = idx->view;
    // filter threshold: every pair whose exact score exceeds `threshold` has a filter score above threshold - eps
    const double eps = (double)filter_rel_eps(X.dtype, X.filt_dtype, X.dtype, X.d) * (double)X.max_norm * (double)X.max_norm;
    const float thr_lo = (float)((double)threshold - eps - 1e-7 * fabs((double)threshold));
    DevBuf cand_i, cand_j, ver_i, ver_j, counters;
    auto cleanup = [&]() { cand_i.release(); cand_j.release(); ver_i.release(); ver_j.release(); counters.release(); };
    int rc = counters.ensure(64);
    if (rc != B2_OK) { cleanup(); return rc; }
    unsigned long long* d_cnt = counters.as<unsigned long long>();
    unsigned long long cand_cap = (unsigned long long)std::max<int64_t>(1 << 20, std::min<int64_t>(idx->n * 8, (int64_t)1 << 28));
    unsigned long long found = 0;
    for (int attempt = 0; attempt < 3; ++attempt) {
        if ((rc = cand_i.ensure(cand_cap * sizeof(int32_t))) != B2_OK || (rc = cand_j.ensure(cand_cap * sizeof(int32_t))) != B2_OK) { cleanup(); return rc; }
        if (cudaMemsetAsync(d_cnt, 0, 16, st) != cudaSuccess) { cleanup(); set_error("memset failed"); return B2_ECUDA; }
        rc = launch_pair_filter(X, thr_lo, part, nparts, cand_i.as<int32_t>(), cand_j.as<int32_t>(), d_cnt, cand_cap, idx->device, st);
        if (rc != B2_OK) { cleanup(); return rc; }
        if (cudaMemcpyAsync(&found, d_cnt, sizeof(found), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess) {
            set_error("pair filter failed on the device: %s", cudaGetErrorString(cudaGetLastError()));
            cleanup();
            return B2_ECUDA;
        }
        if (found <= cand_cap) break;
        cand_cap = found + found / 8 + 1024;  // the candidate buffer overflowed: rerun with the exact size
    }
    if (found > cand_cap) { cleanup(); set_error("pair candidate buffer overflow (%llu)", found); return B2_ENOMEM; }
    unsigned long long kept = 0;
    std::vector<int32_t> hi, hj;
    if (found > 0) {
        if ((rc = ver_i.ensure(found * sizeof(int32_t))) != B2_OK || (rc = ver_j.ensure(found * sizeof(int32_t))) != B2_OK) { cleanup(); return rc; }
        const int64_t blocks = std::min<int64_t>(ceil_div((int64_t)found * 32, 256), 148 * 16);
        pair_verify_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const char*>(X.store), X.dtype, X.d, cand_i.as<int32_t>(),
                                                             cand_j.as<int32_t>(), (int64_t)found, threshold, ver_i.as<int32_t>(),
                                                             ver_j.as<int32_t>(), d_cnt + 1);
        g_stats[ST_LAUNCHES]++;
        g_stats[ST_RESCORED] += (int64_t)found;
        if (cudaGetLastError() != cudaSuccess || cudaMemcpyAsync(&kept, d_cnt + 1, sizeof(kept), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess) {
            set_error("pair verification failed on the device: %s", cudaGetErrorString(cudaGetLastError()));
            cleanup();
            return B2_ECUDA;
        }
        hi.resize(kept);
        hj.resize(kept);
        if (kept) {
            cudaMemcpy(hi.data(), ver_i.p, kept * sizeof(int32_t), cudaMemcpyDeviceToHost);
            cudaMemcpy(hj.data(), ver_j.p, kept * sizeof(int32_t), cudaMemcpyDeviceToHost);
        }
    }
    cleanup();
    // bookkeeping on the host: order the (already exact) pair list by (i, j)
    std::vector<uint64_t> keys(kept);
    for (size_t t = 0; t < kept; ++t) keys[t] = ((uint64_t)(uint32_t)hi[t] << 32) | (uint32_t)hj[t];
    std::sort(keys.begin(), keys.end());
    *n_pairs = (int64_t)kept;
    const int64_t w = std::min<int64_t>(cap, (int64_t)kept);
    for (int64_t t = 0; t < w; ++t) {
        out_i[t] = (int64_t)(keys[t] >> 32);
        out_j[t] = (int64_t)(keys[t] & 0xffffffffu);
    }
    if ((int64_t)kept > cap) { set_error("pair list holds %llu pairs, capacity %lld", kept, (long long)cap); return B2_ERANGE; }
    return B2_OK;
}

int b2_connected_components(int64_t n, const int64_t* pi, const int64_t* pj, int64_t n_pairs, int32_t device, int64_t* labels) {
    if (n < 0 || n_pairs < 0 || (n > 0 && !labels) || (n_pairs > 0 && (!pi || !pj))) { set_error("bad arguments"); return B2_EINVAL; }
    if (n == 0) return B2_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); set_error("no CUDA device: libb2lotus has no CPU fallback"); return B2_ENODEV; }
    if (device < 0 || device >= ndev) { set_error("device %d out of range", device); return B2_EINVAL; }
    DeviceGuard guard(device);
    DevBuf parent, dpi, dpj, dlab, derr;
    auto cleanup = [&]() { parent.release(); dpi.release(); dpj.release(); dlab.release(); derr.release(); };
    int rc;
    if ((rc = parent.ensure(n * sizeof(int64_t))) != B2_OK || (rc = dlab.ensure(n * sizeof(int64_t))) != B2_OK ||
        (rc = dpi.ensure(std::max<int64_t>(n_pairs, 1) * sizeof(int64_t))) != B2_OK ||
        (rc = dpj.ensure(std::max<int64_t>(n_pairs, 1) * sizeof(int64_t))) != B2_OK || (rc = derr.ensure(16)) != B2_OK) {
        cleanup();
        return rc;
    }
    cudaMemset(derr.p, 0, 4);
    if (n_pairs) {
        cudaMemcpy(dpi.p, pi, n_pairs * sizeof(int64_t), cudaMemcpyHostToDevice);
        cudaMemcpy(dpj.p, pj, n_pairs * sizeof(int64_t), cudaMemcpyHostToDevice);
    }
    const unsigned gn = (unsigned)std::min<int64_t>(ceil_div(n, 256), 148 * 16);
    uf_init_kernel<<<gn, 256>>>(parent.as<int64_t>(), n);
    g_stats[ST_LAUNCHES]++;
    if (n_pairs) {
        const unsigned gm = (unsigned)std::min<int64_t>(ceil_div(n_pairs, 256), 148 * 16);
        uf_union_kernel<<<gm, 256>>>(parent.as<int64_t>(), dpi.as<int64_t>(), dpj.as<int64_t>(), n_pairs, n, reinterpret_cast<int*>(derr.p));
        g_stats[ST_LAUNCHES]++;
    }
    uf_flatten_kernel<<<gn, 256>>>(parent.as<int64_t>(), dlab.as<int64_t>(), n);
    g_stats[ST_LAUNCHES]++;
    int herr = 0;
    cudaError_t e = cudaMemcpy(labels, dlab.p, n * sizeof(int64_t), cudaMemcpyDeviceToHost);
    cudaMemcpy(&herr, derr.p, 4, cudaMemcpyDeviceToHost);
    cleanup();
    if (e != cudaSuccess) { set_error("connected components failed on the device: %s", cudaGetErrorString(e)); return B2_ECUDA; }
    if (herr) { set_error("pair list references a node outside [0, %lld)", (long long)n); return B2_ERANGE; }
    return B2_OK;
}

}  // extern "C"
