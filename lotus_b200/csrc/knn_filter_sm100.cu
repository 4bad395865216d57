// knn_filter_sm100.cu — the dominant kernel: fused Q.K^T (tcgen05 tensor cores, TMEM accumulators,
// TMA-staged operand tiles) + per-query streaming top-KP selection in the epilogue.
//
// Replaces the arithmetic of faiss `Index.search` as called from lotus/vector_store/faiss_vs.py:67,75
// (knn_inner_product / knn_L2sqr: blocked sgemm + heap). The N x Q score matrix is never written to HBM.
//
// Role of this kernel in the exact pipeline (DESIGN.md §Pipeline): it is a FILTER. It computes scores with
// bf16 (or TF32) tensor-core products and fp32 accumulation and keeps, per query and per corpus split,
// the KP > k best candidates plus the value `thr` below which everything was discarded. knn_exact.cu then
// re-scores the candidates in the canonical fp64 order and certifies, with a rigorous error margin, that
// nothing discarded could belong to the true top-k; uncertified queries take the dense exact path.
//
// Kernel shape (default: cta_group::2 CTA pairs; cta_group::1 for a single query tile):
//   a CTA owns 128 queries; a pair computes 256 queries x 256 corpus rows per tile, each CTA staging its own query rows
//   and HALF of the corpus tile. K-block = one 128-byte swizzle row (64 bf16 / 32 tf32), UMMA 256x256x16 (bf16) or
//   x8 (tf32) issued by the leader CTA, fp32 accumulators (128 x 256 per CTA) double-buffered in TMEM (2 x 256 columns).
//   warps 0-3 / 4-7: two epilogue sets; set e drains TMEM stage e (every other corpus tile) into its own candidate
//                    list; thread r <-> query row r <-> TMEM lane r
//   warp 8: TMA producer (one lane)   warp 9: MMA issuer (elect.sync lane)   warp 10: TMEM allocator
//   (producer / issuer carry the highest warp ids: the scheduler favours them over the epilogue warps they share a
//   sub-partition with)
//   smem ring of NSTAGES x (A 16 KB + B 16|32 KB), mbarrier full/empty pairs; tmem_full/tmem_empty pairs.
//   Persistent: one CTA per SM, work item = (query-tile pair, corpus split), query tiles fastest so that co-resident
//   workers stream the same corpus tiles and hit them in L2.
#include <cuda.h>

#include "common.cuh"

namespace b2 {

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_N = 256;
constexpr int STAGE_A_BYTES = BLOCK_M * 128;
constexpr int STAGE_B_BYTES = BLOCK_N * 128;
constexpr int STAGE_BYTES = STAGE_A_BYTES + STAGE_B_BYTES;
// Warp roles. The scheduler arbitrates "highest warp id first" among ready warps of an SM sub-partition (warp % 4), and
// the TMEM lane quarter a warp may read is also warp % 4, so epilogue warps necessarily share sub-partitions with the
// producer and the MMA issuer: give those two the HIGHER ids so a busy epilogue warp never delays an MMA issue.
// top-k kernel: TWO epilogue warp-sets (warps 0-3 and 4-7). Set e owns TMEM accumulator stage e, i.e. every other corpus
//   tile, and its own candidate list, so a tile's epilogue has two MMA-tile times to finish and a slow tile (a flush)
//   no longer stalls the tensor pipe.
constexpr int TOPK_THREADS = 352;  // 11 warps
constexpr int TOPK_PRODUCER_WARP = 8, TOPK_MMA_WARP = 9, TOPK_ALLOC_WARP = 10;
// all-pairs kernel: one epilogue set (its epilogue is a compare per score)
constexpr int NUM_THREADS = 224;
constexpr int PRODUCER_WARP = 4, MMA_WARP = 5, ALLOC_WARP = 6;
constexpr int TMEM_COLS = 512;
constexpr int SMEM_LIMIT = 232448;  // 227 KB
constexpr int FILTER_MAX_K = 1000;  // largest k served by the filter (finalize keeps min(k + 32, 1024) survivors per query)

// pending (not yet merged) candidates per query row and epilogue set: a flush is triggered once any row holds
// PEND_FLUSH of them, checked after each 8-column group, so a row never holds more than PEND_FLUSH - 1 + 8 <= PEND
constexpr int PEND = 16;
constexpr int PEND_FLUSH = 8;
__host__ __device__ constexpr int list_bytes(int kp) { return (kp + 2 * PEND) * BLOCK_M * 8; }
__host__ __device__ constexpr int misc_bytes() { return 2 * BLOCK_N * 4 /*xnorm*/ + 256 /*barriers*/; }
// cta_group::2 (a CTA pair computes 256 queries x 256 corpus rows): each CTA stages its own 128 query rows and HALF of
// the corpus tile, so a stage is 32 KB instead of 48 KB and the corpus bytes per SM drop by half.
__host__ __device__ constexpr int stage_bytes(bool two) { return two ? STAGE_A_BYTES + STAGE_B_BYTES / 2 : STAGE_BYTES; }
__host__ __device__ constexpr int num_stages(int kp, bool two = false) {
    int s = (SMEM_LIMIT - list_bytes(kp) - misc_bytes()) / stage_bytes(two);
    return s > 6 ? 6 : s;
}
__host__ __device__ constexpr int smem_bytes(int kp, bool two = false) {
    return num_stages(kp, two) * stage_bytes(two) + list_bytes(kp) + misc_bytes();
}

// ---- PTX wrappers ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a protocol bug must trap (sticky error the host reports) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    uint32_t spins = 0;
    long long t_start = 0;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity), "r"(20000u)  // suspend-time hint (ns): sleep in hardware instead of spinning
            : "memory");
        if (done) break;
        if ((++spins & 0x3ffu) == 0) {
            const long long now = clock64();
            if (t_start == 0) t_start = now;
            else if (now - t_start > 8000000000LL) {  // ~4 s at 2 GHz: no legitimate wait is longer than microseconds
                printf("b2 knn_filter: mbarrier wait timeout (block %d thread %d)\n", blockIdx.x, threadIdx.x);
                __trap();
            }
        }
    }
}
// spin variant without the suspend hint: the MMA issuer must wake the moment its operands land
__device__ __forceinline__ void mbar_wait_spin(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    uint32_t spins = 0;
    long long t_start = 0;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) break;
        if ((++spins & 0x3ffu) == 0) {
            const long long now = clock64();
            if (t_start == 0) t_start = now;
            else if (now - t_start > 8000000000LL) {
                printf("b2 knn_filter: mbarrier wait timeout (block %d thread %d)\n", blockIdx.x, threadIdx.x);
                __trap();
            }
        }
    }
}
// one lane of a converged warp; lets the compiler keep the tcgen05 operands on the uniform datapath
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
        "elect.sync rx|px, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, px;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
template <bool TF32>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (TF32) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives lane (base+t), columns c..c+31
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- CTA-pair (cta_group::2) variants ------------------------------------------------------------------------
// In a 2-CTA cluster bit 24 of a shared::cluster address selects the CTA of the pair; clearing it addresses the
// same offset in the leader (even) CTA.
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PEER_BIT_MASK) : "memory");
}
// executed by BOTH CTAs: the data lands in the issuing CTA's smem, the transaction bytes are counted on the LEADER's barrier
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar) & PEER_BIT_MASK), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// arrive (once the pair's MMAs retire) on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
template <bool TF32>
__device__ __forceinline__ void tc_mma_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (TF32) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}

// UMMA shared-memory descriptor: K-major operand tile, rows of 128 bytes, SWIZZLE_128B (the layout a
// TMA box {128 B, rows} with CU_TENSOR_MAP_SWIZZLE_128B lands in). 8-row groups are 1024 B apart (SBO).
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
    uint64_t desc = 0;
    desc |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);  // start address, bits [0,14)
    desc |= (uint64_t)1 << 16;                        // leading byte offset (ignored for swizzled K-major)
    desc |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset, bits [32,46)
    desc |= (uint64_t)1 << 46;                        // descriptor version 1 (sm_100)
    desc |= (uint64_t)2 << 61;                        // layout type: SWIZZLE_128B
    return desc;
}
// UMMA instruction descriptor: D fp32, A/B bf16 (1) or tf32 (2), both K-major, M = 128, N = 256. fp16 operands (kind::f16,
// format 0) use the bf16 descriptor with FilterParams::idesc_fmt_xor applied at run time (same instruction, same bytes).
template <bool TF32, int M = BLOCK_M>
__device__ __forceinline__ constexpr uint32_t make_idesc() {
    const uint32_t fmt = TF32 ? 2u : 1u;
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

struct FilterParams {
    const float* xnorm;  // [n], L2 only
    float* cand_score;   // [nq, n_splits, KP]
    int32_t* cand_id;    // [nq, n_splits, KP]
    float* cand_thr;     // [nq, n_splits]
    int32_t nq;
    int32_t n;
    int32_t num_kb;        // K-blocks per tile = ceil(d / elements per 128 B)
    int32_t n_mtiles;      // ceil(nq / 128)
    int32_t n_munits;      // schedulable query units: n_mtiles, or ceil(n_mtiles / 2) CTA pairs in cta_group::2 mode
    int32_t n_splits;
    int32_t top1;             // host-side switch only: the TOP1 kernel variant is launched (k-means assignment)
    int32_t tiles_per_split;  // corpus tiles (of 256 rows) per split
    int32_t units_whole;      // two-phase schedule: the first units_whole query units (a multiple of the worker count) sweep the WHOLE
                              // corpus as one item each (split 0); only the remaining units are cut into n_splits splits
    int32_t n_ntiles;         // ceil(n / 256)
    // all-pairs (dedup) schedule: the query matrix IS the corpus; an item is one query tile sweeping only the corpus tiles
    // that can hold a column j > i (upper triangle). Query tiles are dealt to the `nparts` ranks in GROUPS of pair_group
    // consecutive tiles (group g belongs to rank g % nparts): the CTAs of one rank then walk neighbouring corpus tiles at
    // the same time and share them through L2 (dealing single tiles round-robin spreads the concurrently read corpus
    // window nparts times wider: at 10M x 384 and 8 ranks it reached the L2 size and halved the throughput).
    int32_t pair_mode, part, nparts, pair_group, pair_items;
    int32_t pair_align;  // 1: every tile of a group starts its sweep at the group's first corpus tile (equal sweep lengths
                         // keep the CTAs of a wave on the same corpus tile for the whole launch; costs <= group/2 extra tiles)
    int32_t debug_mode;  // timing experiments only (B2_FILTER_DEBUG): 1 = epilogue drains TMEM but ignores the scores,
                         // 2 = accumulate per-role wait cycles into dbg[]
    unsigned long long* dbg;  // [16] cycle counters (debug_mode 2)
    float pair_thr;                   // emit candidates with filter score > pair_thr
    int32_t* pair_i;                  // [pair_cap]
    int32_t* pair_j;
    unsigned long long* pair_count;   // total candidates found (may exceed pair_cap)
    unsigned long long pair_cap;
    uint32_t idesc_fmt_xor;  // kind::f16 kernels: 0 for bf16 operands, F16_FMT_XOR for fp16 operands
};
constexpr uint32_t F16_FMT_XOR = (1u << 7) | (1u << 10);  // A/B format 1 (bf16) -> 0 (fp16)

struct Ring {
    uint8_t* stage_base;
    uint64_t *full_bar, *empty_bar, *tmem_full, *tmem_empty;
    uint32_t tmem_base;
};

// Persistent schedule. A "worker" is a CTA (or a CTA pair); item = (query unit, corpus split), unit fastest so that
// co-resident workers stream the same corpus tiles and share them in L2.
struct Sched {
    int worker, n_workers, rank;  // rank = CTA rank inside the pair (0 in single-CTA mode)
};
template <bool TWO>
__device__ __forceinline__ Sched make_sched() {
    Sched sc;
    if constexpr (TWO) {
        sc.worker = blockIdx.x >> 1;
        sc.n_workers = gridDim.x >> 1;
        sc.rank = (int)cluster_ctarank();
    } else {
        sc.worker = blockIdx.x;
        sc.n_workers = gridDim.x;
        sc.rank = 0;
    }
    return sc;
}
__device__ __forceinline__ int num_items(const FilterParams& p) {
    if (p.pair_mode) return p.pair_items;
    return p.units_whole + (p.n_munits - p.units_whole) * p.n_splits;
}
template <bool TWO>
__device__ __forceinline__ void item_range(const FilterParams& p, const Sched& sc, int item, int& m_tile, int& split, int& t0,
                                           int& t1) {
    if (p.pair_mode) {
        // units are query tiles (single-CTA mode) or pairs of consecutive query tiles (cta_group::2: the two CTAs of a pair
        // take tiles 2u and 2u+1 and sweep the same corpus tiles)
        const int grp = item / p.pair_group;
        const int first = (grp * p.nparts + p.part) * p.pair_group;
        const int unit = first + (item - grp * p.pair_group);
        m_tile = TWO ? 2 * unit + sc.rank : unit;
        split = 0;
        const int lead_tile = (p.pair_align ? first : unit) * (TWO ? 2 : 1);
        t0 = (lead_tile * BLOCK_M) / BLOCK_N;  // first corpus tile that can contain a column > row
        t1 = p.n_ntiles;
    } else {
        int unit;
        if (item < p.units_whole) {  // phase A: one worker, one unit, every corpus tile (all workers stream the same tiles in step)
            unit = item;
            split = 0;
            t0 = 0;
            t1 = p.n_ntiles;
        } else {  // phase B: the leftover units, unit fastest, cut into n_splits splits to fill the last waves
            const int j = item - p.units_whole, rem = p.n_munits - p.units_whole;
            unit = p.units_whole + j % rem;
            split = j / rem;
            t0 = split * p.tiles_per_split;
            t1 = min(t0 + p.tiles_per_split, p.n_ntiles);
        }
        m_tile = TWO ? 2 * unit + sc.rank : unit;
    }
}

// TMA producer: one elected lane (per CTA) streams (query tile, corpus tile) K-blocks into the smem ring.
template <bool TF32, int NSTAGES, bool TWO>
__device__ __forceinline__ void producer_loop(const CUtensorMap* tmap_q, const CUtensorMap* tmap_x, const FilterParams& p,
                                              const Ring& r, const Sched& sc) {
    constexpr int KB_ELEMS = TF32 ? 32 : 64;  // elements per 128-byte K-block row
    constexpr int SB = stage_bytes(TWO);
    const int n_items = num_items(p);
    int stage = 0;
    uint32_t phase = 0;
    for (int item = sc.worker; item < n_items; item += sc.n_workers) {
        int m_tile, split, t0, t1;
        item_range<TWO>(p, sc, item, m_tile, split, t0, t1);
        for (int t = t0; t < t1; ++t) {
            for (int kb = 0; kb < p.num_kb; ++kb) {
                mbar_wait(&r.empty_bar[stage], phase ^ 1);
                uint8_t* sa = r.stage_base + stage * SB;
                uint8_t* sb = sa + STAGE_A_BYTES;
                const int ka = kb, kx = kb;  // K-block (operand column block) of the query / corpus operand
                if constexpr (TWO) {
                    // the leader's full barrier counts the bytes of BOTH CTAs (2 x 32 KB); only the leader arms it
                    if (sc.rank == 0) mbar_arrive_expect_tx(&r.full_bar[stage], 2 * SB);
                    tma_load_2d_pair(sa, tmap_q, &r.full_bar[stage], ka * KB_ELEMS, m_tile * BLOCK_M);
                    tma_load_2d_pair(sb, tmap_x, &r.full_bar[stage], kx * KB_ELEMS, t * BLOCK_N + sc.rank * (BLOCK_N / 2));
                } else {
                    mbar_arrive_expect_tx(&r.full_bar[stage], SB);
                    tma_load_2d(sa, tmap_q, &r.full_bar[stage], ka * KB_ELEMS, m_tile * BLOCK_M);
                    tma_load_2d(sb, tmap_x, &r.full_bar[stage], kx * KB_ELEMS, t * BLOCK_N);
                }
                if (++stage == NSTAGES) {
                    stage = 0;
                    phase ^= 1;
                }
            }
        }
    }
}

// MMA issuer: the whole warp (of the leader CTA in pair mode) walks the schedule and waits on the barriers; one elected
// lane issues tcgen05.mma for every K-block, accumulating a 128x256 fp32 tile per CTA in TMEM.
template <bool TF32, int NSTAGES, bool TWO>
__device__ __forceinline__ void mma_loop(const FilterParams& p, const Ring& r, const Sched& sc) {
    constexpr uint32_t idesc_c = make_idesc<TF32, TWO ? 2 * BLOCK_M : BLOCK_M>();
    const uint32_t idesc = TF32 ? idesc_c : (idesc_c ^ p.idesc_fmt_xor);
    constexpr int SB = stage_bytes(TWO);
    const int n_items = num_items(p);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    const bool dbg = p.debug_mode == 2;
    long long w_full = 0, w_tmem = 0;
    const long long t_begin = dbg ? clock64() : 0;
    for (int item = sc.worker; item < n_items; item += sc.n_workers) {
        int m_tile, split, t0, t1;
        item_range<TWO>(p, sc, item, m_tile, split, t0, t1);
        for (int t = t0; t < t1; ++t) {
            long long c0 = 0;
            if (dbg) c0 = clock64();
            mbar_wait_spin(&r.tmem_empty[acc], acc_phase ^ 1);
            if (dbg) w_tmem += clock64() - c0;
            tc_fence_after();
            const uint32_t tmem_d = r.tmem_base + acc * BLOCK_N;
            for (int kb = 0; kb < p.num_kb; ++kb) {
                if (dbg) c0 = clock64();
                mbar_wait_spin(&r.full_bar[stage], phase);
                if (dbg) w_full += clock64() - c0;
                __syncwarp();
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t sa = smem_u32(r.stage_base + stage * SB);
                    const uint64_t adesc = make_sw128_desc(sa);
                    const uint64_t bdesc = make_sw128_desc(sa + STAGE_A_BYTES);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        // +32 bytes per UMMA_K step inside the 128-byte swizzle row (start address is in 16 B units)
                        if constexpr (TWO)
                            tc_mma_pair<TF32>(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
                        else
                            tc_mma<TF32>(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
                    }
                    // frees the smem stage (in both CTAs of a pair) when these MMAs retire
                    if constexpr (TWO) tc_commit_pair(&r.empty_bar[stage]);
                    else tc_commit(&r.empty_bar[stage]);
                    // accumulator complete -> epilogue (of both CTAs)
                    if (kb == p.num_kb - 1) {
                        if constexpr (TWO) tc_commit_pair(&r.tmem_full[acc]);
                        else tc_commit(&r.tmem_full[acc]);
                    }
                }
                __syncwarp();
                if (++stage == NSTAGES) {
                    stage = 0;
                    phase ^= 1;
                }
            }
            if (++acc == 2) {
                acc = 0;
                acc_phase ^= 1;
            }
        }
    }
    if (dbg && (threadIdx.x & 31) == 0) {
        atomicAdd(&p.dbg[0], (unsigned long long)(clock64() - t_begin));
        atomicAdd(&p.dbg[1], (unsigned long long)w_full);
        atomicAdd(&p.dbg[2], (unsigned long long)w_tmem);
        atomicAdd(&p.dbg[3], 1ull);
    }
}

// barrier init + TMEM allocation shared by both kernels; returns after the block-wide (cluster-wide) sync
template <int NSTAGES, bool TWO>
__device__ __forceinline__ Ring setup_ring(uint8_t* smem, uint64_t* bars, const CUtensorMap* tmap_q, const CUtensorMap* tmap_x,
                                           int producer_warp, int mma_warp, int alloc_warp) {
    Ring r;
    r.stage_base = smem;
    r.full_bar = bars;
    r.empty_bar = bars + NSTAGES;
    r.tmem_full = bars + 2 * NSTAGES;
    r.tmem_empty = r.tmem_full + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(r.tmem_empty + 2);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    if ((smem_u32(smem) & 1023u) != 0) {
        if (threadIdx.x == 0) printf("b2 knn_filter: dynamic smem base not 1024-aligned\n");
        __trap();
    }
    if (warp == producer_warp && lane == 0) {
        tma_prefetch_desc(tmap_q);
        tma_prefetch_desc(tmap_x);
    }
    if (warp == mma_warp && lane == 0) {
        for (int s = 0; s < NSTAGES; ++s) {
            mbar_init(&r.full_bar[s], 1);   // the (leader's) producer arms it; TMA completes the bytes
            mbar_init(&r.empty_bar[s], 1);  // one tcgen05.commit arrival (multicast to both CTAs in pair mode)
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&r.tmem_full[a], 1);
            mbar_init(&r.tmem_empty[a], TWO ? 8 : 4);  // one arrive per epilogue warp (of both CTAs, on the leader)
        }
        fence_barrier_init();
    }
    if (warp == alloc_warp) {
        if constexpr (TWO) tmem_alloc_pair(tmem_ptr, TMEM_COLS);
        else tmem_alloc(tmem_ptr, TMEM_COLS);
    }
    tc_fence_before();
    if constexpr (TWO) cluster_sync_all();  // peers must see initialised barriers before any remote arrive / TMA
    else __syncthreads();
    tc_fence_after();
    r.tmem_base = *tmem_ptr;
    return r;
}

template <bool TWO>
__device__ __forceinline__ void teardown_ring(const Ring& r, int alloc_warp) {
    tc_fence_before();
    if constexpr (TWO) cluster_sync_all();  // nobody leaves while the peer may still touch its smem / TMEM / barriers
    else __syncthreads();
    if ((threadIdx.x >> 5) == alloc_warp) {
        tc_fence_after();
        if constexpr (TWO) tmem_dealloc_pair(r.tmem_base, TMEM_COLS);
        else tmem_dealloc(r.tmem_base, TMEM_COLS);
    }
}

// Replace-min insertion into the thread's candidate list (column `row` of sc/id, stride BLOCK_M): while slots are
// free just take the next one; once full, overwrite the current minimum and rescan for the new minimum (= threshold).
// Called only from flush_pending, where all 32 lanes of the warp run it in lockstep.
template <int KP>
__device__ __forceinline__ void list_insert(float* sc, int32_t* id, float s, int32_t idx, float& thr, int& minpos) {
    // fill phase (minpos < 0 encodes "-(entries so far) - 1"): slots are free, no scan needed until the list is full
    const bool filling = minpos < 0;
    const int pos = filling ? -minpos - 1 : minpos;
    sc[pos * BLOCK_M] = s;
    id[pos * BLOCK_M] = idx;
    if (filling && pos + 1 < KP) {
        minpos = -(pos + 1) - 1;
        return;  // threshold stays -inf
    }
    // new minimum: four independent (value, position) chains so the shared-memory loads and compares overlap
    static_assert(KP % 4 == 0, "list length must be a multiple of 4");
    float m[4];
    int mp[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        m[c] = sc[c * BLOCK_M];
        mp[c] = c;
    }
#pragma unroll
    for (int p = 4; p < KP; p += 4) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const float v = sc[(p + c) * BLOCK_M];
            if (v < m[c]) {
                m[c] = v;
                mp[c] = p + c;
            }
        }
    }
    // ties keep the lowest position, like the sequential scan
    if (m[1] < m[0] || (m[1] == m[0] && mp[1] < mp[0])) { m[0] = m[1]; mp[0] = mp[1]; }
    if (m[3] < m[2] || (m[3] == m[2] && mp[3] < mp[2])) { m[2] = m[3]; mp[2] = mp[3]; }
    if (m[2] < m[0] || (m[2] == m[0] && mp[2] < mp[0])) { m[0] = m[2]; mp[0] = mp[2]; }
    thr = m[0];
    minpos = mp[0];
}

// Merge every lane's pending candidates into its list. Warp-collective: the loop bound is the warp-wide
// maximum so the 32 lanes (32 different queries) execute their insertions together instead of one lane at a
// time (the divergent version of this cost ~20x more issue slots). Returns (new threshold, position of the minimum).
template <int KP>
__device__ __noinline__ float2 flush_pending(float* my_sc, int32_t* my_id, const float* pend_sc, const int32_t* pend_id,
                                             int cnt, float thr, int minpos) {
    int mx = cnt;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    for (int i = 0; i < mx; ++i) {
        if (i < cnt) {
            const float s = pend_sc[i * BLOCK_M];
            if (s > thr) list_insert<KP>(my_sc, my_id, s, pend_id[i * BLOCK_M], thr, minpos);
        }
        __syncwarp();
    }
    return make_float2(thr, __int_as_float(minpos));
}

// One 32-row x 32-column block of scores (thread = row, v = its 32 scores). One warp-wide OR reduction finds the
// 8-column groups in which ANY row beats its threshold (late in a sweep almost none); an active group runs 8 branch-free
// predicated appends into the row's pending buffer and one vote. The pending buffers are merged into the lists by the
// whole warp in lockstep (flush_pending) once any row holds PEND_FLUSH candidates, so nothing is ever dropped.
template <int KPH, bool IS_L2>
__device__ __forceinline__ void process_chunk32(float (&v)[32], int idx0, int valid, const float* xn, float* my_sc, int32_t* my_id,
                                                float* pend_sc, int32_t* pend_id, float& thr, int& minpos, int& cnt, bool dbg,
                                                long long& dbg_flush, long long& dbg_cols) {
    if (valid <= 0) return;  // warp-uniform
    if constexpr (IS_L2) {
        const float4* xn4 = reinterpret_cast<const float4*>(xn);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 x4 = xn4[j];  // warp-uniform address: broadcast
            v[4 * j + 0] = fmaf(2.f, v[4 * j + 0], -x4.x);
            v[4 * j + 1] = fmaf(2.f, v[4 * j + 1], -x4.y);
            v[4 * j + 2] = fmaf(2.f, v[4 * j + 2], -x4.z);
            v[4 * j + 3] = fmaf(2.f, v[4 * j + 3], -x4.w);
        }
    }
    if (valid < 32) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
            if (j >= valid) v[j] = -INFINITY;
    }
    unsigned mine = 0;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        float m = v[8 * g];
#pragma unroll
        for (int jj = 1; jj < 8; ++jj) m = fmaxf(m, v[8 * g + jj]);
        mine |= (m > thr ? 1u : 0u) << g;
    }
    const unsigned active = __reduce_or_sync(0xffffffffu, mine);
    if (active == 0) return;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        if (!(active & (1u << g))) continue;  // warp-uniform
        // branch-free predicated appends for the 8 columns of an active group (cnt <= PEND_FLUSH - 1 on entry, so the
        // pending buffer cannot overflow), then ONE vote per group decides whether the warp flushes
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
            const float s = v[8 * g + jj];
            if (s > thr) {
                pend_sc[cnt * BLOCK_M] = s;
                pend_id[cnt * BLOCK_M] = idx0 + 8 * g + jj;
                ++cnt;
            }
        }
        if (dbg) dbg_cols += 1;
        if (__any_sync(0xffffffffu, cnt >= PEND_FLUSH)) {
            long long f0 = 0;
            if (dbg) f0 = clock64();
            const float2 fr = flush_pending<KPH>(my_sc, my_id, pend_sc, pend_id, cnt, thr, minpos);
            thr = fr.x;
            minpos = __float_as_int(fr.y);
            cnt = 0;
            if (dbg) dbg_flush += clock64() - f0;
        }
    }
}

// k == 1 specialisation (k-means assignment: a few corpus tiles per item, where the list warm-up of the general epilogue
// costs more than the MMAs): each row keeps its best TWO candidates and the third-best score in registers — no smem lists,
// no pending buffer, no flush. b1 >= b2 >= b3; everything not kept scores <= b3, which is the list's discard bound.
template <bool IS_L2>
__device__ __forceinline__ void process_chunk32_top2(float (&v)[32], int idx0, int valid, const float* xn, float& b1, float& b2,
                                                     float& b3, int32_t& i1, int32_t& i2) {
    if (valid <= 0) return;  // warp-uniform
    if constexpr (IS_L2) {
        const float4* xn4 = reinterpret_cast<const float4*>(xn);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 x4 = xn4[j];
            v[4 * j + 0] = fmaf(2.f, v[4 * j + 0], -x4.x);
            v[4 * j + 1] = fmaf(2.f, v[4 * j + 1], -x4.y);
            v[4 * j + 2] = fmaf(2.f, v[4 * j + 2], -x4.z);
            v[4 * j + 3] = fmaf(2.f, v[4 * j + 3], -x4.w);
        }
    }
    if (valid < 32) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
            if (j >= valid) v[j] = -INFINITY;
    }
    unsigned mine = 0;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        float m = v[8 * g];
#pragma unroll
        for (int jj = 1; jj < 8; ++jj) m = fmaxf(m, v[8 * g + jj]);
        mine |= (m > b3 ? 1u : 0u) << g;
    }
    const unsigned active = __reduce_or_sync(0xffffffffu, mine);
    if (active == 0) return;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        if (!(active & (1u << g))) continue;  // warp-uniform
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
            const float s = v[8 * g + jj];
            const int32_t id = idx0 + 8 * g + jj;
            const bool c3 = s > b3, c2 = s > b2, c1 = s > b1;  // strict: an equal score stays behind the earlier column
            b3 = c2 ? b2 : (c3 ? s : b3);
            i2 = c1 ? i1 : (c2 ? id : i2);
            b2 = c1 ? b1 : (c2 ? s : b2);
            i1 = c1 ? id : i1;
            b1 = c1 ? s : b1;
        }
    }
}

template <int KP, bool IS_L2, bool TF32, bool TWO, bool TOP1 = false>
__global__ void __launch_bounds__(TOPK_THREADS, 1)
knn_filter_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                  const FilterParams p) {
    constexpr int NSTAGES = num_stages(KP, TWO);
    static_assert(NSTAGES >= 2, "not enough shared memory for the operand ring");
    constexpr int KPH = KP / 2;  // candidates kept per (row, epilogue set)
    static_assert(KPH % 4 == 0, "list length must allow float4 write-out");

    extern __shared__ __align__(1024) uint8_t smem[];
    float* list_sc = reinterpret_cast<float*>(smem + NSTAGES * stage_bytes(TWO));  // [2 sets][KPH][BLOCK_M]
    int32_t* list_id = reinterpret_cast<int32_t*>(list_sc + KP * BLOCK_M);
    float* pend_sc_base = reinterpret_cast<float*>(list_id + KP * BLOCK_M);        // [2 sets][PEND][BLOCK_M]
    int32_t* pend_id_base = reinterpret_cast<int32_t*>(pend_sc_base + 2 * PEND * BLOCK_M);
    float* s_xn = reinterpret_cast<float*>(pend_id_base + 2 * PEND * BLOCK_M);     // [2 stages][BLOCK_N]
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_xn + 2 * BLOCK_N);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const Ring ring = setup_ring<NSTAGES, TWO>(smem, bars, &tmap_q, &tmap_x, TOPK_PRODUCER_WARP, TOPK_MMA_WARP, TOPK_ALLOC_WARP);
    const int n_items = num_items(p);
    const Sched sc = make_sched<TWO>();

    if (warp == TOPK_PRODUCER_WARP) {
        if (lane == 0) producer_loop<TF32, NSTAGES, TWO>(&tmap_q, &tmap_x, p, ring, sc);
    } else if (warp == TOPK_MMA_WARP) {
        if (sc.rank == 0) mma_loop<TF32, NSTAGES, TWO>(p, ring, sc);
    } else if (warp < 8) {
        // ===================== epilogue set e: streaming top-KPH per query row over the tiles of TMEM stage e ==========
        const int e = warp >> 2;           // epilogue set == TMEM accumulator stage it drains
        const int quad = warp & 3;         // the TMEM lane quarter this warp may read
        const int row = quad * 32 + lane;  // query row inside the tile == TMEM lane
        const int set_tid = threadIdx.x - e * 128;
        float* my_sc = list_sc + e * KPH * BLOCK_M + row;
        int32_t* my_id = list_id + e * KPH * BLOCK_M + row;
        float* pend_sc = pend_sc_base + e * PEND * BLOCK_M + row;
        int32_t* pend_id = pend_id_base + e * PEND * BLOCK_M + row;
        uint64_t* my_full = &ring.tmem_full[e];
        uint64_t* my_empty = &ring.tmem_empty[e];
        const uint32_t taddr = ring.tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(e * BLOCK_N);
        float* xn_tile = s_xn + e * BLOCK_N;
        uint32_t my_phase = 0;   // parity of the next completion of tmem_full[e]
        uint32_t tile_ctr = 0;   // tiles issued by the MMA warp so far; stage = tile_ctr & 1
        long long epi_wait = 0, dbg_flush = 0, dbg_cols = 0;
        const long long epi_begin = p.debug_mode == 2 ? clock64() : 0;
        for (int item = sc.worker; item < n_items; item += sc.n_workers) {
            int m_tile, split, t0, t1;
            item_range<TWO>(p, sc, item, m_tile, split, t0, t1);
#pragma unroll 4
            for (int i = 0; i < KPH; ++i) {
                my_sc[i * BLOCK_M] = -INFINITY;
                my_id[i * BLOCK_M] = -1;
            }
            float thr = -INFINITY;
            int minpos = -1;  // fill phase, 0 entries (see list_insert)
            int cnt = 0;      // pending candidates of this row
            float b1 = -INFINITY, b2 = -INFINITY, b3 = -INFINITY;  // TOP1: best two scores + discard bound
            int32_t i1 = -1, i2 = -1;
            for (int t = t0; t < t1; ++t, ++tile_ctr) {
                if ((int)(tile_ctr & 1u) != e) continue;  // the other set's tile
                const int col0 = t * BLOCK_N;
                if constexpr (IS_L2) {
                    // stage this tile's squared norms; the 4 warps of the set sync on their own named barrier:
                    // once before overwriting (everyone is done reading the previous tile's norms), once after
                    if (e == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
                    else asm volatile("bar.sync 2, 128;" ::: "memory");
                    for (int c = set_tid; c < BLOCK_N; c += 128) {
                        const int g = col0 + c;
                        xn_tile[c] = g < p.n ? __ldg(p.xnorm + g) : 0.f;
                    }
                    if (e == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
                    else asm volatile("bar.sync 2, 128;" ::: "memory");
                }
                long long e0 = 0;
                if (p.debug_mode == 2) e0 = clock64();
                mbar_wait(my_full, my_phase);
                my_phase ^= 1;
                if (p.debug_mode == 2) epi_wait += clock64() - e0;
                tc_fence_after();
                const int ncols = min(BLOCK_N, p.n - col0);
                // eight 32-column chunks, TMEM loads software-pipelined one chunk ahead (va / vb ping-pong)
                float va[32], vb[32];
                tmem_ld32(taddr, va);
#pragma unroll 1
                for (int h = 0; h < 4; ++h) {
                    tmem_ld_wait();                            // chunk 2h is in va
                    tmem_ld32(taddr + (2 * h + 1) * 32, vb);   // chunk 2h+1 in flight while va is processed
                    if constexpr (TOP1)
                        process_chunk32_top2<IS_L2>(va, col0 + (2 * h) * 32, ncols - (2 * h) * 32, xn_tile + (2 * h) * 32, b1, b2, b3, i1, i2);
                    else if (p.debug_mode != 1)
                        process_chunk32<KPH, IS_L2>(va, col0 + (2 * h) * 32, ncols - (2 * h) * 32, xn_tile + (2 * h) * 32, my_sc, my_id,
                                                    pend_sc, pend_id, thr, minpos, cnt, p.debug_mode == 2, dbg_flush, dbg_cols);
                    tmem_ld_wait();                            // chunk 2h+1 is in vb
                    if (h < 3) {
                        tmem_ld32(taddr + (2 * h + 2) * 32, va);  // next chunk in flight while vb is processed
                    } else {
                        // whole accumulator stage now in registers: hand TMEM back to the (leader's) MMA warp
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            if constexpr (TWO) mbar_arrive_leader(my_empty);
                            else mbar_arrive(my_empty);
                        }
                    }
                    if constexpr (TOP1)
                        process_chunk32_top2<IS_L2>(vb, col0 + (2 * h + 1) * 32, ncols - (2 * h + 1) * 32, xn_tile + (2 * h + 1) * 32, b1, b2, b3,
                                                    i1, i2);
                    else if (p.debug_mode != 1)
                        process_chunk32<KPH, IS_L2>(vb, col0 + (2 * h + 1) * 32, ncols - (2 * h + 1) * 32, xn_tile + (2 * h + 1) * 32, my_sc,
                                                    my_id, pend_sc, pend_id, thr, minpos, cnt, p.debug_mode == 2, dbg_flush, dbg_cols);
                    else if (vb[0] == 12345.678f) thr = va[1] + vb[1];  // keep the loads alive in the timing experiment
                }
            }
            if constexpr (TOP1) {
                // same [KPH] list layout as the general epilogue: two real entries, the rest stays (-inf, -1)
                my_sc[0 * BLOCK_M] = b1;
                my_id[0 * BLOCK_M] = i1;
                my_sc[1 * BLOCK_M] = b2;
                my_id[1 * BLOCK_M] = i2;
                thr = b3;
            } else {
                const float2 fr = flush_pending<KPH>(my_sc, my_id, pend_sc, pend_id, cnt, thr, minpos);
                thr = fr.x;
                minpos = __float_as_int(fr.y);
                cnt = 0;
            }
            // write this (query, split, set) candidate list
            const int q = m_tile * BLOCK_M + row;
            if (q < p.nq) {
                const size_t lidx = ((size_t)q * p.n_splits + split) * 2 + e;
                float4* osc = reinterpret_cast<float4*>(p.cand_score + lidx * KPH);
                int4* oid = reinterpret_cast<int4*>(p.cand_id + lidx * KPH);
#pragma unroll 4
                for (int i = 0; i < KPH / 4; ++i) {
                    osc[i] = make_float4(my_sc[(4 * i + 0) * BLOCK_M], my_sc[(4 * i + 1) * BLOCK_M],
                                         my_sc[(4 * i + 2) * BLOCK_M], my_sc[(4 * i + 3) * BLOCK_M]);
                    oid[i] = make_int4(my_id[(4 * i + 0) * BLOCK_M], my_id[(4 * i + 1) * BLOCK_M],
                                       my_id[(4 * i + 2) * BLOCK_M], my_id[(4 * i + 3) * BLOCK_M]);
                }
                p.cand_thr[lidx] = thr;  // -inf unless this list overflowed
            }
        }
        if (p.debug_mode == 2 && lane == 0) {
            atomicAdd(&p.dbg[4], (unsigned long long)(clock64() - epi_begin));
            atomicAdd(&p.dbg[5], (unsigned long long)epi_wait);
            atomicAdd(&p.dbg[6], 1ull);
            atomicAdd(&p.dbg[7], (unsigned long long)dbg_flush);
            atomicAdd(&p.dbg[8], (unsigned long long)dbg_cols);
        }
    }

    teardown_ring<TWO>(ring, TOPK_ALLOC_WARP);
}

// ---- all-pairs threshold filter (sem_dedup): same mainloop, the epilogue emits (i, j) candidates -------------------
constexpr int PAIR_STAGES = 4;
constexpr int PAIR_SMEM = PAIR_STAGES * STAGE_BYTES + 256;
constexpr int PAIR_STAGES_TWO = 6;  // cta_group::2: 32 KB per stage and CTA (A 16 KB + half of B)
constexpr int PAIR_SMEM_TWO = PAIR_STAGES_TWO * stage_bytes(true) + 256;

template <bool TF32, bool TWO>
__global__ void __launch_bounds__(NUM_THREADS, 1)
pair_filter_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x, const FilterParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    constexpr int NST = TWO ? PAIR_STAGES_TWO : PAIR_STAGES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NST * stage_bytes(TWO));
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const Ring ring = setup_ring<NST, TWO>(smem, bars, &tmap_q, &tmap_x, PRODUCER_WARP, MMA_WARP, ALLOC_WARP);
    const int n_items = num_items(p);
    const Sched sc = make_sched<TWO>();
    if (warp == PRODUCER_WARP) {
        if (lane == 0) producer_loop<TF32, NST, TWO>(&tmap_q, &tmap_x, p, ring, sc);
    } else if (warp == MMA_WARP) {
        if (sc.rank == 0) mma_loop<TF32, NST, TWO>(p, ring, sc);  // the leader issues for the pair
    } else if (warp < 4) {
        const int quad = warp;  // epilogue warps 0-3: TMEM quarter == warp id
        const int row = quad * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        const float thr = p.pair_thr;
        for (int item = sc.worker; item < n_items; item += sc.n_workers) {
            int m_tile, split, t0, t1;
            item_range<TWO>(p, sc, item, m_tile, split, t0, t1);
            const int gi = m_tile * BLOCK_M + row;  // global row of this thread
            for (int t = t0; t < t1; ++t) {
                const int col0 = t * BLOCK_N;
                mbar_wait(&ring.tmem_full[acc], acc_phase);
                tc_fence_after();
                const uint32_t taddr = ring.tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BLOCK_N);
#pragma unroll 1
                for (int c = 0; c < BLOCK_N / 32; ++c) {
                    float v[32];
                    tmem_ld32(taddr + c * 32, v);
                    tmem_ld_wait();
                    if (c == BLOCK_N / 32 - 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            if constexpr (TWO) mbar_arrive_leader(&ring.tmem_empty[acc]);  // 4 warps x 2 CTAs arrive on the leader
                            else mbar_arrive(&ring.tmem_empty[acc]);
                        }
                    }
                    float mx = v[0];
#pragma unroll
                    for (int j = 1; j < 32; ++j) mx = fmaxf(mx, v[j]);
                    if (mx > thr && gi < p.n) {
                        const int idx0 = col0 + c * 32;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int gj = idx0 + j;
                            if (v[j] > thr && gj > gi && gj < p.n) {  // strict upper triangle, inside the matrix
                                const unsigned long long pos = atomicAdd(p.pair_count, 1ull);
                                if (pos < p.pair_cap) {
                                    p.pair_i[pos] = gi;
                                    p.pair_j[pos] = gj;
                                }
                            }
                        }
                    }
                }
                if (++acc == 2) {
                    acc = 0;
                    acc_phase ^= 1;
                }
            }
        }
    }
    teardown_ring<TWO>(ring, ALLOC_WARP);
}

// ---- host side ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p) {
        set_error("cuTensorMapEncodeTiled is not available from the driver (%s)", cudaGetErrorString(e));
        return nullptr;
    }
    fn = reinterpret_cast<PFN_encodeTiled>(p);
    return fn;
}

// 2-D row-major matrix [rows, cols] with `pitch` elements per row; box = {128 bytes of K, box_rows rows}
int make_tmap(CUtensorMap* map, const void* base, int dtype, int64_t rows, int64_t cols, int64_t pitch, int box_rows) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return B2_ECUDA;
    const int esz = dtype == B2_F32 ? 4 : 2;
    const CUtensorMapDataType ttype = dtype == B2_F32   ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                      : dtype == B2_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                        : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)pitch * esz};
    cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (gstride[0] & 15) != 0) {
        set_error("TMA operand not 16-byte aligned (base %p, pitch %lld B)", base, (long long)gstride[0]);
        return B2_EINVAL;
    }
    CUresult r = enc(map, ttype, 2,
                     const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows %lld cols %lld pitch %lld)", (int)r,
                  (long long)rows, (long long)cols, (long long)pitch);
        return B2_ECUDA;
    }
    return B2_OK;
}

template <int KP, bool IS_L2, bool TF32, bool TWO, bool TOP1 = false>
int launch_variant(const CUtensorMap& tq, const CUtensorMap& tx, const FilterParams& p, int grid, cudaStream_t stream) {
    auto kern = knn_filter_kernel<KP, IS_L2, TF32, TWO, TOP1>;
    constexpr int smem = smem_bytes(KP, TWO);
    // the attribute is per DEVICE (not per process): set it on every launch — a microsecond — so that a process driving
    // several B200s (B200VS(device=i) for several i) launches correctly on each of them
    B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(TOPK_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = TWO ? 2 : 1;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    B2_CUDA(cudaLaunchKernelEx(&cfg, kern, tq, tx, p));
    B2_LAUNCH_CHECK();
    g_stats[ST_FILTER_LAUNCHES]++;
    return B2_OK;
}

template <int KP, bool TWO>
int launch_kp(bool is_l2, bool tf32, const CUtensorMap& tq, const CUtensorMap& tx, const FilterParams& p, int grid,
              cudaStream_t stream) {
    if constexpr (KP == 16) {
        if (p.top1) {  // k == 1: register-resident top-2 epilogue
            if (is_l2) {
                return tf32 ? launch_variant<KP, true, true, TWO, true>(tq, tx, p, grid, stream)
                            : launch_variant<KP, true, false, TWO, true>(tq, tx, p, grid, stream);
            }
            return tf32 ? launch_variant<KP, false, true, TWO, true>(tq, tx, p, grid, stream)
                        : launch_variant<KP, false, false, TWO, true>(tq, tx, p, grid, stream);
        }
    }
    if (is_l2) {
        return tf32 ? launch_variant<KP, true, true, TWO>(tq, tx, p, grid, stream)
                    : launch_variant<KP, true, false, TWO>(tq, tx, p, grid, stream);
    }
    return tf32 ? launch_variant<KP, false, true, TWO>(tq, tx, p, grid, stream)
                : launch_variant<KP, false, false, TWO>(tq, tx, p, grid, stream);
}

template <bool TWO>
int launch_two(int kp, bool is_l2, bool tf32, const CUtensorMap& tq, const CUtensorMap& tx, const FilterParams& p, int grid,
               cudaStream_t stream) {
    switch (kp) {
        case 16: return launch_kp<16, TWO>(is_l2, tf32, tq, tx, p, grid, stream);
        case 32: return launch_kp<32, TWO>(is_l2, tf32, tq, tx, p, grid, stream);
        case 64: return launch_kp<64, TWO>(is_l2, tf32, tq, tx, p, grid, stream);
        case 96: return launch_kp<96, TWO>(is_l2, tf32, tq, tx, p, grid, stream);
        default: set_error("internal: unsupported candidate capacity %d", kp); return B2_EINVAL;
    }
}

int sm_count(int device) {
    static int cached[64] = {0};
    if (device >= 0 && device < 64 && cached[device]) return cached[device];
    int n = 148;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device);
    if (device >= 0 && device < 64) cached[device] = n;
    return n;
}

}  // namespace

int filter_kp_for_k(int k) {
    if (k <= 6) return 16;
    if (k <= 16) return 32;
    if (k <= 40) return 64;
    if (k <= FILTER_MAX_K) return 96;  // k > 64: several corpus splits share the load, see filter_min_splits_for_k
    return 0;
}

// k > 64 does not fit one candidate list (96 entries = 2 epilogue sets x 48 is what shared memory allows next to the operand
// ring), so the corpus is cut into enough splits that each (split, set) sub-list expects at most ~24 of a query's top k —
// half its capacity, 4-5 standard deviations of headroom for rows in random order. A sub-list that overflows anyway is caught
// by the certificate (its discard bound reaches the k-th exact score) and that query takes the dense path.
int filter_min_splits_for_k(int k) { return k <= 64 ? 1 : (int)ceil_div(k, 48); }

// cta_group::2 (CTA pairs) needs at least two query tiles; B2_FILTER_2CTA=0/1 overrides the default.
bool filter_use_pair(int64_t nq) {
    static int mode = -1;
    if (mode < 0) {
        const char* e = getenv("B2_FILTER_2CTA");
        mode = e ? (atoi(e) != 0 ? 1 : 0) : 1;  // default: CTA pairs
    }
    return mode == 1 && ceil_div(nq, BLOCK_M) >= 2;
}

// Number of corpus splits: enough work items to fill the machine, and few idle workers in the last wave.
// In pair mode a worker is a CTA pair and a query unit is two query tiles.
int filter_choose_splits(int64_t nq, int64_t n, int num_sms, bool two_cta, bool top1, int min_splits, int* units_whole) {
    if (units_whole) *units_whole = 0;
    {
        static int forced = -1;  // B2_FILTER_SPLITS: experiments only
        if (forced < 0) {
            const char* e = getenv("B2_FILTER_SPLITS");
            forced = e ? atoi(e) : 0;
        }
        if (forced > 0) {
            const int64_t nt = ceil_div(n, BLOCK_N);
            int s = (int)std::min<int64_t>(forced, nt);
            while (s > 1 && ceil_div(nt, ceil_div(nt, s)) != s) --s;
            return s;
        }
    }
    const int64_t n_mtiles = ceil_div(nq, BLOCK_M);
    const int64_t n_units = two_cta ? ceil_div(n_mtiles, 2) : n_mtiles;
    const int64_t workers = two_cta ? std::max(1, num_sms / 2) : num_sms;
    const int64_t n_ntiles = ceil_div(n, BLOCK_N);
    // cost model (measured, profiles/README.md): an item costs its corpus tiles plus ~13 tile-times of list warm-up, the
    // kernel takes `waves` such items back to back, and every extra split adds two candidate lists per query to finalize
    const double kWarmupTiles = top1 ? 1.0 : 13.0;  // the register-resident top-2 epilogue has no list to warm up
    double best_cost = 1e300;
    int best = 0;
    for (int s = std::max(1, min_splits); s <= 256 && s <= n_ntiles; ++s) {
        const int64_t tps = ceil_div(n_ntiles, s);
        if (ceil_div(n_ntiles, tps) != s) continue;  // every split must receive tiles
        const int64_t items = n_units * s;
        const int64_t waves = ceil_div(items, workers);
        const double cost = (double)waves * ((double)tps + kWarmupTiles) * (1.0 + 0.004 * s);
        if (cost < best_cost - 1e-9) {
            best_cost = cost;
            best = s;
        }
    }
    // Two-phase schedule: as many whole waves as possible run ONE unit per worker over the whole corpus (one list warm-up per
    // wave instead of one per split, and the workers still stream the same corpus tiles in step, which is what keeps them in
    // L2); only the leftover units (< one per worker) are cut into splits, just fine enough to fill the last waves. On a
    // 125k-row shard with 100k queries: 5 x (489 + 13) + 2 x (70 + 13) = 2676 tile-times against 16 x (163 + 13) = 2816.
    static const bool two_phase_on = [] { const char* e = getenv("B2_FILTER_TWO_PHASE"); return e ? atoi(e) != 0 : true; }();
    const int64_t waves_a = n_units / workers;
    if (units_whole && two_phase_on && min_splits <= 1 && waves_a >= 1) {
        const int64_t ua = waves_a * workers, rem = n_units - ua;
        const double cost_a = (double)waves_a * ((double)n_ntiles + kWarmupTiles);
        double best2 = 1e300;
        int s2 = 1;
        if (rem == 0) {
            best2 = cost_a;
        } else {
            for (int s = 1; s <= 256 && s <= n_ntiles; ++s) {
                const int64_t tps = ceil_div(n_ntiles, s);
                if (ceil_div(n_ntiles, tps) != s) continue;
                const int64_t waves_b = ceil_div(rem * s, workers);
                const double cost = (cost_a + (double)waves_b * ((double)tps + kWarmupTiles)) * (1.0 + 0.002 * s);
                if (cost < best2 - 1e-9) {
                    best2 = cost;
                    s2 = s;
                }
            }
        }
        if (best2 < best_cost - 1e-9) {
            *units_whole = (int)ua;
            return s2;
        }
    }
    return best;
}

int launch_knn_filter(const MatView& X, const void* q_filt, int64_t q_pitch, int64_t nq, int metric, int kp,
                      int n_splits, bool two_cta, float* cand_score, int32_t* cand_id, float* cand_thr, int device,
                      cudaStream_t stream, bool top1, int units_whole) {
    if (nq <= 0 || X.n <= 0) return B2_OK;
    if (X.n > 0x7fffff00LL || nq > 0x7fffff00LL) {
        set_error("matrix too large for 32-bit row ids (n=%lld nq=%lld)", (long long)X.n, (long long)nq);
        return B2_ERANGE;
    }
    const bool tf32 = X.filt_dtype == B2_F32;
    const int kb_elems = tf32 ? 32 : 64;
    CUtensorMap tq, tx;
    const int64_t op_cols = X.d;
    B2_TRY(make_tmap(&tq, q_filt, X.filt_dtype, nq, op_cols, q_pitch, BLOCK_M));
    // pair mode: each CTA of the pair loads HALF of the 256-row corpus tile
    B2_TRY(make_tmap(&tx, X.filt, X.filt_dtype, X.n, op_cols, X.filt_pitch, two_cta ? BLOCK_N / 2 : BLOCK_N));
    FilterParams p;
    p.idesc_fmt_xor = X.filt_dtype == B2_F16 ? F16_FMT_XOR : 0u;
    p.xnorm = X.norm2;
    p.cand_score = cand_score;
    p.cand_id = cand_id;
    p.cand_thr = cand_thr;
    p.nq = (int32_t)nq;
    p.n = (int32_t)X.n;
    p.num_kb = (int32_t)ceil_div(X.d, kb_elems);
    p.n_mtiles = (int32_t)ceil_div(nq, BLOCK_M);
    p.n_munits = two_cta ? (p.n_mtiles + 1) / 2 : p.n_mtiles;
    p.n_ntiles = (int32_t)ceil_div(X.n, BLOCK_N);
    p.tiles_per_split = (int32_t)ceil_div(p.n_ntiles, n_splits);
    p.n_splits = n_splits;
    p.units_whole = units_whole;
    p.top1 = (top1 && kp == 16) ? 1 : 0;  // register-resident top-2 epilogue: requested by the k-means assignment path only
    p.pair_mode = 0;
    p.part = 0;
    p.nparts = 1;
    {
        static int dbg = -1;
        if (dbg < 0) {
            const char* e = getenv("B2_FILTER_DEBUG");
            dbg = e ? atoi(e) : 0;
        }
        p.debug_mode = dbg;
    }
    static unsigned long long* dbg_dev = nullptr;
    p.dbg = nullptr;
    if (p.debug_mode == 2) {
        if (!dbg_dev) cudaMalloc(&dbg_dev, 16 * sizeof(unsigned long long));
        cudaMemsetAsync(dbg_dev, 0, 16 * sizeof(unsigned long long), stream);
        p.dbg = dbg_dev;
    }
    p.pair_thr = 0.f;
    p.pair_i = p.pair_j = nullptr;
    p.pair_count = nullptr;
    p.pair_cap = 0;
    if ((int64_t)p.tiles_per_split * (n_splits - 1) >= p.n_ntiles) {
        set_error("internal: empty corpus split (tiles %d, splits %d)", p.n_ntiles, n_splits);
        return B2_EINVAL;
    }
    if (units_whole < 0 || units_whole > p.n_munits) {
        set_error("internal: bad two-phase schedule (%d whole units of %d)", units_whole, p.n_munits);
        return B2_EINVAL;
    }
    const int64_t items = (int64_t)units_whole + (int64_t)(p.n_munits - units_whole) * n_splits;
    if (units_whole > 0 && n_splits > 1) {
        // whole units write split 0 only: the other lists of their queries must read as empty (id -1, bound -inf)
        B2_CUDA(cudaMemsetAsync(cand_id, 0xFF, (size_t)nq * n_splits * kp * sizeof(int32_t), stream));
        B2_TRY(launch_fill_f32(cand_thr, nq * (int64_t)n_splits * 2, -INFINITY, stream));
    }
    const bool is_l2 = metric == B2_METRIC_L2;
    if (is_l2 && !X.norm2) {
        set_error("internal: L2 filter without row norms");
        return B2_EINVAL;
    }
    int rc;
    if (two_cta) {
        const int pairs = (int)std::min<int64_t>(items, sm_count(device) / 2);
        rc = launch_two<true>(kp, is_l2, tf32, tq, tx, p, 2 * pairs, stream);
    } else {
        const int grid = (int)std::min<int64_t>(items, sm_count(device));
        rc = launch_two<false>(kp, is_l2, tf32, tq, tx, p, grid, stream);
    }
    if (rc == B2_OK && p.debug_mode == 2) {
        unsigned long long h[16];
        cudaStreamSynchronize(stream);
        cudaMemcpy(h, p.dbg, sizeof(h), cudaMemcpyDeviceToHost);
        const double nm = h[3] ? (double)h[3] : 1.0, ne = h[6] ? (double)h[6] : 1.0;
        fprintf(stderr,
                "[b2 filter dbg] mma warps=%llu: total %.3e cyc, wait_full %.1f%%, wait_tmem_empty %.1f%% | epilogue warps=%llu: total "
                "%.3e cyc, wait_tmem_full %.1f%%, in flush %.1f%%, active columns/warp %.3e\n",
                h[3], h[0] / nm, 100.0 * h[1] / (double)(h[0] ? h[0] : 1), 100.0 * h[2] / (double)(h[0] ? h[0] : 1), h[6], h[4] / ne,
                100.0 * h[5] / (double)(h[4] ? h[4] : 1), 100.0 * h[7] / (double)(h[4] ? h[4] : 1), h[8] / ne);
    }
    return rc;
}

// query tiles per dealing group of the all-pairs schedule: one per SM, so that one wave of CTAs is one group
// (B2_PAIR_GROUP overrides it; the tests use a small value to exercise the dealing on small matrices)
static int pair_group_size(int device) {
    const char* e = getenv("B2_PAIR_GROUP");
    if (e && atoi(e) > 0) return atoi(e);
    return sm_count(device);
}

// All pairs i < j of X whose filter inner product exceeds thr (sem_dedup). Candidates land in pair_i/pair_j (device,
// capacity cap) in arbitrary order; *pair_count receives the total found.
int launch_pair_filter(const MatView& X, float thr, int part, int nparts, int32_t* pair_i, int32_t* pair_j,
                       unsigned long long* pair_count, unsigned long long cap, int device, cudaStream_t stream) {
    if (X.n <= 1) return B2_OK;
    if (X.n > 0x7fffff00LL) {
        set_error("matrix too large for 32-bit row ids (n=%lld)", (long long)X.n);
        return B2_ERANGE;
    }
    const bool tf32 = X.filt_dtype == B2_F32;
    const int kb_elems = tf32 ? 32 : 64;
    CUtensorMap tq, tx;
    B2_TRY(make_tmap(&tq, X.filt, X.filt_dtype, X.n, X.d, X.filt_pitch, BLOCK_M));
    B2_TRY(make_tmap(&tx, X.filt, X.filt_dtype, X.n, X.d, X.filt_pitch, BLOCK_N));
    FilterParams p;
    memset(&p, 0, sizeof(p));
    p.idesc_fmt_xor = X.filt_dtype == B2_F16 ? F16_FMT_XOR : 0u;
    p.nq = (int32_t)X.n;
    p.n = (int32_t)X.n;
    p.num_kb = (int32_t)ceil_div(X.d, kb_elems);
    static const bool two = [] { const char* e = getenv("B2_PAIR_2CTA"); return e ? atoi(e) != 0 : true; }();  // default: CTA pairs
    const bool two_cta = two && ceil_div(X.n, BLOCK_M) >= 2;
    if (two_cta) B2_TRY(make_tmap(&tx, X.filt, X.filt_dtype, X.n, X.d, X.filt_pitch, BLOCK_N / 2));  // each CTA stages half a corpus tile
    p.n_mtiles = (int32_t)ceil_div(X.n, BLOCK_M);
    p.n_munits = two_cta ? (p.n_mtiles + 1) / 2 : p.n_mtiles;
    p.n_ntiles = (int32_t)ceil_div(X.n, BLOCK_N);
    p.n_splits = 1;
    p.tiles_per_split = p.n_ntiles;
    p.pair_mode = 1;
    p.debug_mode = 0;
    p.dbg = nullptr;
    p.part = part;
    p.nparts = nparts;
    p.pair_group = two_cta ? std::max(1, pair_group_size(device) / 2) : pair_group_size(device);  // one unit per worker
    {
        const char* e = getenv("B2_PAIR_ALIGN");
        p.pair_align = e ? (atoi(e) != 0) : 1;  // measured (scripts/pair_sched_exp.py): +15 % at 1M rows, neutral at 10M x 8 ranks
    }
    p.pair_thr = thr;
    p.pair_i = pair_i;
    p.pair_j = pair_j;
    p.pair_count = pair_count;
    p.pair_cap = cap;
    // this rank's query tiles: the full groups g = part (mod nparts) plus the trailing partial group if it is ours (it is
    // then this rank's last group, so item -> tile stays a closed form)
    const int64_t full_groups = p.n_munits / p.pair_group, rem = p.n_munits % p.pair_group;
    const int64_t my_full = full_groups > part ? ceil_div(full_groups - part, (int64_t)nparts) : 0;
    const int64_t items = my_full * p.pair_group + ((rem && full_groups % nparts == part) ? rem : 0);
    p.pair_items = (int32_t)items;
    if (items <= 0) return B2_OK;
    if (two_cta) {
        const int pairs = (int)std::min<int64_t>(items, sm_count(device) / 2);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(2 * pairs));
        cfg.blockDim = dim3(NUM_THREADS);
        cfg.dynamicSmemBytes = PAIR_SMEM_TWO;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        if (tf32) {
            B2_CUDA(cudaFuncSetAttribute(pair_filter_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PAIR_SMEM_TWO));
            B2_CUDA(cudaLaunchKernelEx(&cfg, pair_filter_kernel<true, true>, tq, tx, p));
        } else {
            B2_CUDA(cudaFuncSetAttribute(pair_filter_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PAIR_SMEM_TWO));
            B2_CUDA(cudaLaunchKernelEx(&cfg, pair_filter_kernel<false, true>, tq, tx, p));
        }
    } else {
        const int grid = (int)std::min<int64_t>(items, sm_count(device));
        if (tf32) {
            B2_CUDA(cudaFuncSetAttribute(pair_filter_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PAIR_SMEM));
            pair_filter_kernel<true, false><<<grid, NUM_THREADS, PAIR_SMEM, stream>>>(tq, tx, p);
        } else {
            B2_CUDA(cudaFuncSetAttribute(pair_filter_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PAIR_SMEM));
            pair_filter_kernel<false, false><<<grid, NUM_THREADS, PAIR_SMEM, stream>>>(tq, tx, p);
        }
    }
    B2_LAUNCH_CHECK();
    g_stats[ST_FILTER_LAUNCHES]++;
    return B2_OK;
}

}  // namespace b2
