// wisecondor_b200 - shared device/host helpers (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include <string>
#include <vector>
#include <algorithm>
#include "../../include/wisecondor_b200.h"

// ---- error plumbing -----------------------------------------------------------------------------------
void wc_set_error(const char* fmt, ...);

#define WC_CUDA(expr)                                                                                   \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) {                                                                        \
            wc_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__);   \
            return WC_ERR_CUDA;                                                                         \
        }                                                                                               \
    } while (0)

#define WC_CHECK_ARG(cond)                                                                              \
    do {                                                                                                \
        if (!(cond)) {                                                                                  \
            wc_set_error("bad argument: %s (%s:%d)", #cond, __FILE__, __LINE__);                        \
            return WC_ERR_ARG;                                                                          \
        }                                                                                               \
    } while (0)

// ---- context ------------------------------------------------------------------------------------------
// Grow-only device workspace: the search/test paths ask for named slots; memory is reused across calls.
struct wc_buf {
    void* p = nullptr;
    size_t bytes = 0;
};

enum { WC_NBUF = 56, WC_NPHASE = 12, WC_NCOUNTER = 12 };

// Workspace slots (one grow-only device buffer each).
enum {
    SLOT_XC = 0, SLOT_NORMS, SLOT_ROWCS, SLOT_ROWCE, SLOT_RBMETA, SLOT_CAND_D, SLOT_CAND_J, SLOT_SEGCNT,
    SLOT_SEGFLAG, SLOT_SLOW, SLOT_SCRATCH, SLOT_IO_X, SLOT_IO_IDX, SLOT_IO_DIST, SLOT_ROWTHR,
    SLOT_IN_KEY, SLOT_IN_J, SLOT_IN_CNT, SLOT_N32, SLOT_F16STAT,                                                             // search
    SLOT_PROF = 20, SLOT_PIV_IDS = 21, SLOT_PIV_X = 22, SLOT_PIV_N = 23, SLOT_PIV_META = 37, SLOT_S_STACK = 38,
    SLOT_T_COPY = 24, SLOT_T_ZT, SLOT_T_RT, SLOT_T_NT, SLOT_T_SD, SLOT_T_FLAGS, SLOT_T_TOTALS, SLOT_T_PROJ,   // test
    SLOT_T_REVCNT = 44, SLOT_T_REVCUR, SLOT_T_DIRTY, SLOT_T_PAIRS,
    SLOT_S_ZC = 32, SLOT_S_META, SLOT_S_STATUS, SLOT_S_RC, SLOT_S_AUX,                                                       // segmentation
    SLOT_P_FIRST = 40,                                                                                 // newref prep
    SLOT_FIN_J = 48, SLOT_FIN_D, SLOT_FIN_P, SLOT_FIN_GRP,                                             // K6 split form: shortlists, exact distances, work list
    SLOT_WIDE_D = 52, SLOT_WIDE_ROWS                                                                   // wide-refsize search: chunk distances, exclusion ranges
};

// State of a sharded symmetric search between its three calls (wc_newref_shard_begin / _sweep / _finish).
struct wc_shard_plan {
    int valid = 0;
    int N = 0, S = 0, k = 0, cap = 0, in_cap = 0, world = 1, rank = 0;
    int nb = 0, bp = 0, b0 = 0, b1 = 0;          // blocks of 128 bins: all, per rank, this rank's [b0, b1)
    int row0 = 0, row1 = 0, rows_per = 0;        // this rank's bins [row0, row1) (row1 <= N), bins per rank (padded)
    int nkc = 0, nd_last = 0, extra_h = 0, ld = 0, nstages = 0, nrb = 0, nseg = 0, gridA = 0, gridB = 0;
    size_t Npad = 0, smem = 0, nlistA = 0;
    long long tilesA = 0, tilesB = 0, tiles_plain = 0;
    double mcoef = 0.0, madd = 0.0;              // margins of the filter (fp64: madd = 0; fp16: see wc_newref_topk)
    int f16 = 0, ldh = 0;                        // fp16 tensor-core filter in use (1 mma.sync, 2 tcgen05), its padded sample count
    int pivots = 0;                              // pivots of the K5t pivot pass (0: none)
    const double* corrected = nullptr;
    const unsigned long long* thr = nullptr;     // the threshold table handed to wc_newref_shard_sweep
    int stage = 0;                               // 1 after begin, 2 after sweep
};

struct wc_ctx {
    int device = 0;
    int sm_count = 0;
    wc_buf buf[WC_NBUF];
    cudaEvent_t ev[2 * WC_NPHASE];
    double phase_ms[WC_NPHASE];
    long long counter[WC_NCOUNTER];
    const int* zs_npairs_d = nullptr;    // device counters of the last wc_zscore_batch: listed pairs of pass 1..repeats-1
    int zs_repeats = 0;
    long long zs_pair_limit = 0, zs_all_pairs = 0;
    // wc_newref_topk_host: where the search may start copying the first half of its table while the second half is re-scored
    int32_t* d2h_idx_h = nullptr; double* d2h_dist_h = nullptr; size_t d2h_rows_done = 0;
    cudaStream_t d2h_stream = nullptr; cudaEvent_t d2h_ev = nullptr;
    void* search_plan = nullptr;         // host plan of the last search (wc_search.cu: SearchPlan), freed through search_plan_free
    void (*search_plan_free)(void*) = nullptr;
    unsigned long long sched_hash = 0;   // fingerprint of the K5 schedule metadata currently on the device
    unsigned timed_mask = 0;        // phases whose event pair is recorded but not yet read (asynchronous calls)
    int k5_stages = 0;              // 0 = automatic TMA ring depth
    int k5_group = 0;               // CTAs sharing a row block per scheduling round of K5 (0 = automatic)
    int k5_sym = 8;                 // symmetric search: 0 = off, f >= 2 = on with 1/f of the block pairs in the first pass
    int k5_f16 = 2;                 // filter of K5: 0 fp64 (DMMA), 1 fp16 on mma.sync (HMMA), 2 fp16 on tcgen05 / TMEM (UTCHMMA)
    int k5_f16_checked = 1;         // 1: K4h's fp16 range check is read at the end of the call (no sync before K5), 0: right after K4h
    int k5_pivots = 1;              // K5t: pivot pass before a symmetric search (0 = off)
    unsigned long long piv_hash = 0;   // fingerprint of the pivot pass' piece table on the device
    float* dbg_scores = nullptr;    // wc_debug_filter_scores: where K5t dumps its filter distances (caller-owned), or NULL
    int dbg_ld = 0;
    const int* k6_stats_d = nullptr;   // device counters of the last split K6: [0] live entries, [1] shortlisted candidates
    int k6_g4 = 0;                  // K6c: 1 = candidate rows four per TMA request (tile::gather4) instead of one bulk copy each (measured: no faster)
    int k6_parts = 4;               // wc_newref_topk_host: row ranges K6 runs in (all but the last copied to the host while the next is re-scored)
    int k6_select = 1;              // K6a: 1 = streaming histogram select (entries never held), 0 = bisection on entries held in shared memory
    int k6_split = 1;               // K6: 1 = select -> streaming re-score (bulk copies) -> rank, 0 = fused kernel
    int k6_chunk = 0, k6_warps = 0, k6_prod = 0;     // K6c tuning: samples per chunk, consumer / producer warps (0 = default)
    int k5_lag = 0;                 // chunks the trailing consumer warps of K5 lag behind the leading ones
    int debug_profile = 0;          // K5 writes per-CTA cycle counters when set (wc_debug_profile)
    void* encode_tiled = nullptr;   // cuTensorMapEncodeTiled, resolved through the runtime (no -lcuda)
    wc_shard_plan shard;            // the sharded symmetric search in flight on this context, if any
};

int wc_reserve(wc_ctx* ctx, int slot, size_t bytes, void** out);

// ---- small PTX wrappers ----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Non-blocking probe of a phase (mbarrier.test_wait never suspends the thread).
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// 2-D TMA tile load, global -> shared, completion on an mbarrier (SASS: UTMALDG).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
// Shared-space 64-bit load from a 32-bit shared address.  `volatile` only pins its order against the mbarrier
// wait at the NVVM level; ptxas still schedules the resulting ld.shared freely among the DMMAs.
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void lds_v2f64(uint32_t addr, double& v0, double& v1) {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v0), "=d"(v1) : "r"(addr));
}
// FP64 tensor-core MMA, D(8x8) += A(8x4) * B(4x8)   (SASS: DMMA.8x8x4)
__device__ __forceinline__ void dmma_8x8x4(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ double ld_cg_f64(const double* p) {
    double v;
    asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ int ld_cg_s32(const int* p) {
    int v;
    asm volatile("ld.global.cg.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
