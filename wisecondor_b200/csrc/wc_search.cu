// wisecondor_b200 - newref reference-bin search on B200 (sm_100a).
//
// Replaces getReference / getRefForBins (/root/reference/wisetools.py:364-398, 298-325): for every target bin,
// the squared Euclidean distance over samples to every bin on the other chromosomes, keeping the `refsize`
// smallest ordered by (distance, index).
//
// Kernels
//   K4 wc_prepare_kernel      X' = X - 1 (padded, TMA-friendly), n_i = sum_s X'[i][s]^2, and two extra "samples"
//                             per row, (1, -n_i/2), so that the contraction itself yields the score
//                             s_ij = X'_i.X'_j - (n_i + n_j)/2 = -d~_ij/2                                (HBM bound)
//   K5 wc_dist_topk_kernel    fp64 tensor-core contraction (DMMA.8x8x4) on 128x128 tiles, operands staged by TMA
//                             (SWIZZLE_128B) through an mbarrier ring, fused with a streaming per-row threshold
//                             filter on the raw accumulator bits: only entries that can still be among the row's
//                             k smallest leave the SM.  The distance matrix never exists.              (FP64 bound)
//   K6 wc_finalize_kernel     per row: shortlist = entries within an error margin of the k-th smallest d~, exact
//                             re-score in the reference's operation order, rank by (d, index), remap to
//                             other-chromosome coordinates                                              (L2 bound)
//   K6b wc_exhaustive_kernel  exact brute force for rows the streaming path could not bound (massive ties)
//
// Why the filter works on integer bit patterns: on B200 plain FP64 instructions (DADD/DSETP/DFMA) share the FP64
// pipe with DMMA and are starved ~20x while another warp of the same SM sub-partition streams DMMAs (measured,
// tools/dmma_coissue.cu); integer and shared-memory instructions are not.  With the score in the accumulator,
// "d~ <= tau" is one unsigned 64-bit compare per entry, and the candidate buffers, the prune and the emission
// path need no FP64 arithmetic at all.
#include "wc_common.cuh"
#include <cuda_fp16.h>

namespace {

typedef unsigned long long u64;

constexpr int BM = 128;             // target rows per CTA tile
constexpr int BN = 128;             // candidate columns per CTA tile
constexpr int BK = 16;              // samples per pipeline stage (16 doubles = one 128-byte swizzle row)
constexpr int CONSUMER_WARPS = 8;   // each warp owns 16 rows x 128 cols of the tile: no cross-warp state
constexpr int CONSUMER_THREADS = CONSUMER_WARPS * 32;
constexpr int WROWS = BM / CONSUMER_WARPS;   // 16 rows per warp
constexpr int PRODUCER_WARPS = 4;   // one warp group; only warp 0 lane 0 issues TMA, the group donates registers
constexpr int TOPK_THREADS = CONSUMER_THREADS + PRODUCER_WARPS * 32;
constexpr int TILE_BYTES = BM * BK * 8;               // 16 KiB per operand per stage
constexpr int STAGE_BYTES = 2 * TILE_BYTES;
constexpr int MAX_STAGES = 6;
constexpr int HIST_BINS = 256;
constexpr int FIN_THREADS = 128;    // one thread per shortlisted candidate during the exact re-score
constexpr int FIN_CHUNK = 32;       // samples staged per pipeline step of the re-score
constexpr int FIN_BUCKETS = 1024;   // locality buckets of the re-score's work list
constexpr int FIN_ECAP = 1360;      // candidate entries of one row K6 collects in shared memory (16 KiB; later the target's own row: S <= 2040); more: read from the sources
constexpr int EXH_THREADS = 256;
constexpr int STG = 128;            // per-warp staging entries for column-side candidates (symmetric pass)
constexpr u64 KEY_NEVER = 0ull;     // threshold key of an inactive row: no finite negative score passes

// Shared memory of K5: [nstages x STAGE_BYTES operand ring, 1024-byte aligned][TopkState][8 warps x scratch]
struct __align__(16) TopkState {
    uint64_t full[MAX_STAGES];
    uint64_t empty[MAX_STAGES];
    uint64_t gate;       // opened by the leading warps after `lag` chunks; the lagging warps start behind it
    u64 thr[BM];         // per-row threshold key = bits(-tau/2); an entry passes iff bits(score) <= thr (unsigned)
    double nrm[BM];      // n_i
    int cnt[BM];         // entries in the row's candidate buffer
    unsigned char flag[BM];   // 1 = buffer could not be bounded -> exhaustive fallback
    int stg_cnt[CONSUMER_WARPS];   // symmetric pass: column-side candidates staged by each warp
};

struct TopkArgs {
    const double* norms;     // [Npad]
    const int* row_cs;       // [N]
    const int* row_ce;       // [N]
    int N;
    int row_begin, row_end;
    int nkc;                 // k chunks of BK, the last one holding the two extra samples
    int nd_last;             // data double-steps (8 samples each) in the last chunk: 0 or 1
    int extra_h;             // 8-sample block of the last chunk that holds (1, -n/2)
    const int* rb_skip_lo;       // [nrb] first skipped column tile (own chromosome interior)
    const int* rb_skip_n;        // [nrb] number of skipped column tiles
    int nrb;
    const int* cta_piece_begin;  // [grid+1] this CTA's pieces are [begin, end)
    const int* pieces;           // [npieces][5]: row block, first valid-tile index, end, step, segment id
    u64* cand_key;               // [nseg][BM][cap] score bit patterns
    int* cand_j;
    int* seg_cnt;                // [nseg][BM]
    int* seg_flag;               // [nseg][BM]
    int cap;
    int k;
    double mcoef;                // margin(v) = mcoef * (n_i + |v|)
    double tau_init;
    long long* prof;             // optional [grid][8] per-CTA cycle counters (consumer warp 0), or nullptr
    long long* trace;            // optional debug timeline of CTA 0: [2 warps (0 and 4)][64 tiles][4 stamps]
    u64* row_thr;                // [rows] tightest threshold key any CTA has found for the row (shared between segments)
    int lag;                     // chunks by which warps 4-7 trail warps 0-3 (0 = all in phase)
    int nstages;                 // depth of the TMA ring (3..MAX_STAGES)
    // --- symmetric search (each unordered pair of bin blocks contracted once), see the host side ---
    const int* tile_list;        // list mode: the column tile of every list entry (nullptr: arithmetic progression mode)
    const int* rb_list_off;      // [nrb] first list entry of the row block; a piece's q indexes the list from there
    int final_prune;             // 1: prune and publish every row's threshold when a piece ends
    u64* in_key;                 // [Nrows][in_cap] candidates found for a bin while it was on the COLUMN side of a tile
    int* in_j;
    int* in_cnt;                 // [Nrows] entries offered (may exceed in_cap: the row then takes the exact fallback)
    int in_cap;
    const u64* col_thr;          // thresholds indexed by GLOBAL bin (== row_thr when the launch starts at row 0)
    double madd;                 // margin(v) = mcoef * (n_i + |v|) + madd  (0 for the fp64 filter)
    const double* madd_p;        // when set: madd lives on the device (written by wc_f16_margin_kernel - no host round trip)
    int kb_last;                 // K5t: column of the B operand's last 64-sample chunk (folded norms: its second version)
    const float* n32;            // fp16 filter: the bins' squared norms in fp32, +inf for padding rows
    const float* coln32;         // K5t: norms of the COLUMN rows (== n32, or the pivot matrix' norms in the pivot pass)
    const int* col_ids;          // K5t pivot pass: global bin of every row of the pivot matrix (nullptr: columns are bins)
    float* dbg;                  // debug (K5t, DBG instantiation): every filter distance d~ lands in dbg[row - row_begin][column]
    int dbg_ld;
};

__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ u64 warp_min_u64(u64 v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { u64 t = __shfl_xor_sync(0xffffffffu, v, o); v = t < v ? t : v; }
    return v;
}
__device__ __forceinline__ u64 warp_max_u64(u64 v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { u64 t = __shfl_xor_sync(0xffffffffu, v, o); v = t > v ? t : v; }
    return v;
}
__device__ __forceinline__ void cp_async_8(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// 256-bit read-only streaming load (SASS LDG.E.NA.256.CONSTANT): four consecutive doubles, no L1 allocation, the rest of
// the 256-byte block prefetched into L2 (DRAM sees 256-byte requests: the rows of a matrix beyond the L2 are gathered at random)
__device__ __forceinline__ void ldg_nc_v4f64(const double* p, double& a, double& b, double& c, double& d) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
__device__ __forceinline__ void sts_v2f64(uint32_t addr, double v0, double v1) {
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(v0), "d"(v1) : "memory");
}
__device__ __forceinline__ int bucket_of(double d, double mn, float scale) {
    int b = (int)((float)(d - mn) * scale);
    return b < 0 ? 0 : (b > HIST_BINS - 1 ? HIST_BINS - 1 : b);
}
// threshold key for "d~ <= tau": bits(-tau/2); tau is kept strictly positive so the key has its sign bit set and
// every score >= +0 (d~ <= 0, rounding noise of duplicates) passes the unsigned compare.
__device__ __forceinline__ u64 key_of_tau(double tau) { return (u64)__double_as_longlong(-0.5 * tau); }
inline u64 host_key_of_tau(double tau) {
    const double v = -0.5 * tau;
    u64 bits;
    memcpy(&bits, &v, sizeof(bits));
    return bits;
}
__device__ __forceinline__ double dist_of_key(u64 key) { return -2.0 * __longlong_as_double((long long)key); }
template <typename Args>
__device__ __forceinline__ double madd_of(const Args& a) { return a.madd_p != nullptr ? __ldg(a.madd_p) : a.madd; }

// Warp-collective prune of one row's candidate buffer, on score keys (unsigned order == distance order).  The
// buffer is copied once into the warp's shared scratch with independent L2 loads; an integer bisection finds a
// cut with k <= #{key <= cut} <= k + 24 (about 5 rounds on real data); v* = the largest key <= cut bounds the row's
// final k-th smallest distance from above, and everything within the error margin of it is written back compacted.
// Integer-only apart from the five FP64 operations that turn v* into the new threshold.
template <int PER_LANE>   // cap / 32: every load of the buffer is issued before the first one is consumed
__device__ __noinline__ void prune_row(u64* ck, int* cj, int n, int k, double nrm, double mcoef, double madd, int lane,
                                       u64* sk, int* sj, u64* thr_out, int* n_out) {
    // The row's buffer lives in registers for the whole prune (16 or 32 keys + column ids per lane; the accumulators
    // are dead between tiles): the bisection counts, the v* search and the compaction never touch memory again.
    (void)sk; (void)sj;
    u64 d[PER_LANE];
    int j[PER_LANE];
#pragma unroll
    for (int t = 0; t < PER_LANE; ++t) {
        const int i = t * 32 + lane;
        d[t] = i < n ? __ldcg(ck + i) : ~0ull;       // padding never counts (keys <= mid < ~0) and is never kept
        j[t] = i < n ? __ldcg(cj + i) : 0;
    }
    u64 lo = ~0ull, hi = 0ull;
#pragma unroll
    for (int t = 0; t < PER_LANE; ++t) {
        if (t * 32 + lane < n) {
            lo = d[t] < lo ? d[t] : lo;
            hi = d[t] > hi ? d[t] : hi;
        }
    }
    lo = warp_min_u64(lo);
    hi = warp_max_u64(hi);
    const int k_hi = k + 24;
    u64 blo = lo, bhi = hi, cut = hi;           // count(<= cut) >= k throughout
    int c_hi = n;
    for (int it = 0; it < 70 && c_hi > k_hi; ++it) {
        if (bhi - blo < 2) break;               // bracket exhausted (ties): keep the current cut
        const u64 mid = blo + ((bhi - blo) >> 1);
        int c = 0;
#pragma unroll
        for (int t = 0; t < PER_LANE; ++t) c += d[t] <= mid ? 1 : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (c >= k) { bhi = mid; c_hi = c; cut = mid; } else { blo = mid; }
    }
    u64 vstar = 0ull;
#pragma unroll
    for (int t = 0; t < PER_LANE; ++t)
        if (d[t] <= cut && d[t] > vstar) vstar = d[t];
    vstar = warp_max_u64(vstar);
    const double dv = dist_of_key(vstar);
    double tau = dv + mcoef * (nrm + fabs(dv)) + madd;
    const double tiny = fmax(mcoef * nrm, 1e-300);
    if (!(tau > tiny)) tau = tiny;
    const u64 thr = key_of_tau(tau);
    int w = 0;
#pragma unroll
    for (int t = 0; t < PER_LANE; ++t) {
        const bool keep = d[t] <= thr && t * 32 + lane < n;
        const unsigned km = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            const int pos = w + __popc(km & ((1u << lane) - 1u));
            ck[pos] = d[t];
            cj[pos] = j[t];
        }
        w += __popc(km);
    }
    __syncwarp();
    *thr_out = thr;
    *n_out = w;
}

// ---------------------------------------------------------------------------------------------------------
// K5: score tiles on the FP64 tensor cores + streaming top-k filter
// ---------------------------------------------------------------------------------------------------------
// SYM = true: besides the row-side filter, every score is also tested against the threshold of its COLUMN's bin and
// offered to that bin's incoming buffer - the tile (I, J) then serves the row blocks I and J, and (J, I) is never computed.
template <bool SYM>
__global__ void __launch_bounds__(TOPK_THREADS, 1)
wc_dist_topk_kernel(const __grid_constant__ CUtensorMap tmap, const TopkArgs a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    if (smem_u32(smem_raw) & 1023u) __trap();   // SWIZZLE_128B tiles need a 1024-byte aligned base
    const int STAGES = a.nstages;
    unsigned char* tiles = smem_raw;
    TopkState& sm = *reinterpret_cast<TopkState*>(smem_raw + (size_t)STAGES * STAGE_BYTES);
    unsigned char* scratch = reinterpret_cast<unsigned char*>(&sm + 1);
    const int tid = threadIdx.x;
    const int warp_all = tid >> 5, lane = tid & 31;
    const int warp = warp_all - PRODUCER_WARPS;     // consumer warp index (negative in the producer group)

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&sm.full[s], 1);
            mbar_init(&sm.empty[s], CONSUMER_WARPS);
        }
        mbar_init(&sm.gate, CONSUMER_WARPS / 2);
        for (int w = 0; w < CONSUMER_WARPS; ++w) sm.stg_cnt[w] = 0;
        mbar_fence_init();
        tma_prefetch_desc(&tmap);
    }
    __syncthreads();

    // this CTA's work: a list of pieces (row block, arithmetic progression of its valid column tiles), see the host side
    const int pb = a.cta_piece_begin[blockIdx.x], pe = a.cta_piece_begin[blockIdx.x + 1];
    if (pb >= pe) return;

    if (warp_all < PRODUCER_WARPS) {
        // ===== TMA producer: one elected lane streams the A (target rows) and B (candidate rows) k-slices =====
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        if (warp_all == 0 && lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int pi = pb; pi < pe; ++pi) {
                const int* pc = a.pieces + (size_t)pi * 5;
                const int rbp = pc[0], q1 = pc[2], qs = pc[3];
                const int skip_lo = a.rb_skip_lo[rbp], skip_n = a.rb_skip_n[rbp];
                const int* tl = a.tile_list ? a.tile_list + a.rb_list_off[rbp] : nullptr;
                const int row0 = a.row_begin + rbp * BM;
                for (int q = pc[1]; q < q1; q += qs) {
                    const int t = tl ? tl[q] : (q < skip_lo ? q : q + skip_n);
                    const int col0 = t * BN;
                    for (int kc = 0; kc < a.nkc; ++kc) {
                        mbar_wait(&sm.empty[stage], phase ^ 1u);
                        mbar_arrive_expect_tx(&sm.full[stage], STAGE_BYTES);
                        tma_load_2d(tiles + (size_t)stage * STAGE_BYTES, &tmap, kc * BK, row0, &sm.full[stage]);
                        tma_load_2d(tiles + (size_t)stage * STAGE_BYTES + TILE_BYTES, &tmap, kc * BK, col0, &sm.full[stage]);
                        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
        return;
    }

    // ===== consumers: 8 warps; warp w owns rows [16w, 16w+16) x all 128 columns = 2 x 16 DMMA tiles =====
    // Rows are warp-private, so the threshold / candidate-count state needs no CTA-level barrier: each warp runs
    // its own epilogue and prune and drifts from the others by at most the depth of the TMA ring.
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");

    // Fragment <-> tile mapping.  A DMMA.8x8x4 lane (g = lane/4, q = lane%4) supplies A[g][q] and B[q][g].  Rows of an
    // 8-row group are visited in the order perm(g) = (g&1)*4 + (g>>1) and each lane fetches 16 bytes = two
    // consecutive samples (k = 8h+2q, 8h+2q+1), used as the q-th sample of two successive MMAs.  Both operands
    // use the same sample permutation, so the dot products are unchanged; with the TMA 128-byte swizzle
    // (16-byte chunk index ^= row & 7) every quarter-warp of an LDS.128 then touches 128 distinct bytes of
    // banks: no conflicts.
    const int g = lane >> 2, q4 = lane & 3;
    const int pg = ((g & 1) << 2) | (g >> 1);
    const uint32_t a_off = (uint32_t)(warp * WROWS + pg) * 128u;
    const uint32_t b_off = (uint32_t)TILE_BYTES + (uint32_t)pg * 128u;
    uint32_t sw[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) sw[h] = (uint32_t)(((4 * h + q4) ^ pg) << 4);
    const uint32_t swx = a.extra_h ? sw[1] : sw[0];

    const uint32_t tiles_u32 = smem_u32(tiles);
    const size_t scratch_per_warp = (size_t)a.cap * 12 > 8192 ? (size_t)a.cap * 12 : 8192;
    u64* w_sk = reinterpret_cast<u64*>(scratch + (size_t)warp * scratch_per_warp);
    int* w_sj = reinterpret_cast<int*>(w_sk + a.cap);
    // SYM: this warp's copy of the 128 column-side thresholds of the current tile (after the 8 scratch areas)
    u64* w_ct = reinterpret_cast<u64*>(scratch + (size_t)CONSUMER_WARPS * scratch_per_warp) + warp * BN;
    // SYM: column-side candidates (key, bin j, candidate i) wait here until a warp-wide flush appends them to the bins'
    // incoming buffers - 32 global atomics in flight at once instead of one round trip per entry
    uint4* w_stg = reinterpret_cast<uint4*>(scratch + (size_t)CONSUMER_WARPS * scratch_per_warp +
                                            (size_t)CONSUMER_WARPS * BN * sizeof(u64)) + warp * STG;
    int* w_stgc = &sm.stg_cnt[warp];
    const int r0w = warp * WROWS;               // first tile row of this warp
    u64* w_thr = sm.thr + r0w;
    double* w_nrm = sm.nrm + r0w;
    int* w_cnt = sm.cnt + r0w;
    unsigned char* w_flag = sm.flag + r0w;
    int my_cs[2] = {0, 0}, my_ce[2] = {0, 0};   // excluded column range [cs, ce) of this lane's two rows
    int stage = 0;
    uint32_t phase = 0;
    const size_t seg_stride = (size_t)BM * a.cap;
    bool ready = false;

    // Optional phase offset between the two consumer warps of every SM sub-partition (warps w and w+4 share one).
    const bool leader = warp < CONSUMER_WARPS / 2;
    int gate_left = (leader && a.lag > 0) ? a.lag : -1;      // chunks until this leader opens the gate
    if (!leader && a.lag > 0) mbar_wait(&sm.gate, 0);

    long long pf_wait = 0, pf_epi = 0, pf_prune = 0, pf_nprune = 0, pf_emit = 0;
    const long long pf_t0 = clock64();
    int pi = pb;
    const int* pc = a.pieces + (size_t)pi * 5;
    int rb = pc[0], q = pc[1], q1 = pc[2], qs = pc[3], seg = pc[4];
    int skip_lo = a.rb_skip_lo[rb], skip_n = a.rb_skip_n[rb];
    const int* tl = a.tile_list ? a.tile_list + a.rb_list_off[rb] : nullptr;
    bool new_piece = true;

    // Prune the rows named in `need` (a warp-uniform mask over the warp's 16 rows): tighten and publish their thresholds.
    auto prune_rows = [&](unsigned need, u64* ck, int* cj) {
        while (need) {
            const int rw = __ffs(need) - 1;
            need &= need - 1;
            int n = w_cnt[rw];
            if (n > a.cap) n = a.cap;
            u64 thr;
            int kept;
            ++pf_nprune;
            u64* rk = ck + (size_t)(r0w + rw) * a.cap;
            int* rj = cj + (size_t)(r0w + rw) * a.cap;
            __threadfence_block();
            if (a.cap <= 512)
                prune_row<16>(rk, rj, n, a.k, w_nrm[rw], a.mcoef, madd_of(a), lane, w_sk, w_sj, &thr, &kept);
            else
                prune_row<32>(rk, rj, n, a.k, w_nrm[rw], a.mcoef, madd_of(a), lane, w_sk, w_sj, &thr, &kept);
            if (lane == 0) {
                if (kept > a.cap - BN) {       // a tie plateau wider than the buffer: exact fallback
                    w_flag[rw] = 1;
                    w_thr[rw] = KEY_NEVER;
                    w_cnt[rw] = 0;
                } else {
                    const int row = a.row_begin + rb * BM + r0w + rw;
                    const u64 other = atomicMin(a.row_thr + (row - a.row_begin), thr);   // publish; adopt a tighter one
                    w_thr[rw] = other < thr ? other : thr;
                    w_cnt[rw] = kept;
                }
            }
            __syncwarp();
        }
    };
    auto flush_incoming = [&]() {
        __syncwarp();
        int n = *w_stgc;
        if (n > STG) n = STG;
        for (int e = lane; e < n; e += 32) {
            const uint4 v = w_stg[e];
            const int j = (int)v.z;
            const int w = atomicAdd(a.in_cnt + j, 1);
            if (w < a.in_cap) {
                a.in_key[(size_t)j * a.in_cap + w] = ((u64)v.y << 32) | (u64)v.x;
                a.in_j[(size_t)j * a.in_cap + w] = (int)v.w;
            }
        }
        __syncwarp();
        if (lane == 0) *w_stgc = 0;
        __syncwarp();
    };
    int tcount = 0;                             // tiles done by this CTA (debug timeline index)
    while (true) {
        if (q >= q1) {
            // piece finished: flush this warp's rows of its segment, move to the next piece
            __syncwarp();
            if (SYM) flush_incoming();
            if (a.final_prune) {
                // every row leaves its best threshold behind: the bins on the column side of later tiles are filtered by it
                const unsigned need = __ballot_sync(0xffffffffu, lane < WROWS && w_cnt[lane] > a.k + 24 &&
                                                                     w_cnt[lane] <= a.cap && !w_flag[lane]);
                prune_rows(need, a.cand_key + (size_t)seg * seg_stride, a.cand_j + (size_t)seg * seg_stride);
            }
            if (lane < WROWS) {
                a.seg_cnt[(size_t)seg * BM + r0w + lane] = w_cnt[lane] > a.cap ? a.cap : w_cnt[lane];
                a.seg_flag[(size_t)seg * BM + r0w + lane] = w_flag[lane];
            }
            if (++pi >= pe) break;
            pc = a.pieces + (size_t)pi * 5;
            rb = pc[0]; q = pc[1]; q1 = pc[2]; qs = pc[3]; seg = pc[4];
            skip_lo = a.rb_skip_lo[rb]; skip_n = a.rb_skip_n[rb];
            tl = a.tile_list ? a.tile_list + a.rb_list_off[rb] : nullptr;
            new_piece = true;
            continue;
        }
        if (new_piece) {
            new_piece = false;
            __syncwarp();
            if (lane < WROWS) {
                const int row = a.row_begin + rb * BM + r0w + lane;
                const bool valid = row < a.row_end;
                w_nrm[lane] = valid ? a.norms[row] : 0.0;
                // a threshold found by any other CTA for this row (other columns) bounds the row's k-th distance too
                w_thr[lane] = valid ? __ldcg(a.row_thr + (row - a.row_begin)) : KEY_NEVER;
                w_cnt[lane] = 0;
                w_flag[lane] = 0;
            }
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                const int row = a.row_begin + rb * BM + r0w + mt * 8 + pg;
                const bool valid = row < a.row_end;
                my_cs[mt] = valid ? a.row_cs[row] : 0;
                my_ce[mt] = valid ? a.row_ce[row] : 0;
            }
            __syncwarp();
        }
        const int t = tl ? tl[q] : (q < skip_lo ? q : q + skip_n);
        const int col0 = t * BN;
        q += qs;
        if (SYM) {
            // the column bins' published thresholds (L2 -> this warp's shared copy), landed long before the epilogue
            __syncwarp();                           // the previous tile's epilogue has finished reading the copy
            cp_async_16(w_ct + 2 * lane, a.col_thr + col0 + 2 * lane);
            cp_async_16(w_ct + 64 + 2 * lane, a.col_thr + col0 + 64 + 2 * lane);
            cp_async_commit();
        }
        u64 shared_thr = ~0ull;                 // issued now, consumed after the tile's MMAs: latency fully hidden
        if (lane < WROWS) {
            const int row = a.row_begin + rb * BM + r0w + lane;
            if (row < a.row_end) shared_thr = __ldcg(a.row_thr + (row - a.row_begin));
        }
        const bool tr_on = a.trace != nullptr && blockIdx.x == 0 && (warp & 3) == 0 && lane == 0 && tcount < 64;
        long long* tr = tr_on ? a.trace + ((size_t)(warp >> 2) * 64 + tcount) * 4 : nullptr;
        ++tcount;
        if (tr_on) tr[0] = clock64();

        double acc[2][16][2];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int nt = 0; nt < 16; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;

        for (int kc = 0; kc < a.nkc; ++kc) {
            if (!ready) {
                const long long pf_w0 = clock64();
                mbar_wait(&sm.full[stage], phase);
                pf_wait += clock64() - pf_w0;
            }
            const uint32_t base = tiles_u32 + (uint32_t)stage * STAGE_BYTES;
            // probe the next stage's barrier now; the answer is only needed after this chunk's DMMAs
            int nstage = stage + 1;
            uint32_t nphase = phase;
            if (nstage == STAGES) { nstage = 0; nphase ^= 1u; }
            const bool ready_next = mbar_test_wait(&sm.full[nstage], nphase);
            const bool last = kc == a.nkc - 1;
            const int nd = last ? a.nd_last : 2;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (h < nd) {
                    double fa[2][2];
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) lds_v2f64(base + a_off + mt * 1024 + sw[h], fa[mt][0], fa[mt][1]);
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        double fb[8][2];
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            lds_v2f64(base + b_off + (half * 8 + i) * 1024 + sw[h], fb[i][0], fb[i][1]);
#pragma unroll
                        for (int u = 0; u < 2; ++u)
#pragma unroll
                            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                                for (int i = 0; i < 8; ++i)
                                    dmma_8x8x4(acc[mt][half * 8 + i][0], acc[mt][half * 8 + i][1], fa[mt][u], fb[i][u]);
                    }
                }
            }
            if (last) {
                // The two extra samples (1, -n/2) sit in one 16-byte slot of the row.  Feeding the B operand with
                // the pair swapped makes the step add 1*(-n_j/2) + (-n_i/2)*1 to the dot product.
                double fa[2][2];
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) lds_v2f64(base + a_off + mt * 1024 + swx, fa[mt][0], fa[mt][1]);
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    double fb[8][2];
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        lds_v2f64(base + b_off + (half * 8 + i) * 1024 + swx, fb[i][0], fb[i][1]);
#pragma unroll
                    for (int u = 0; u < 2; ++u)
#pragma unroll
                        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                            for (int i = 0; i < 8; ++i)
                                dmma_8x8x4(acc[mt][half * 8 + i][0], acc[mt][half * 8 + i][1], fa[mt][u], fb[i][1 - u]);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.empty[stage]);
            if (gate_left > 0 && --gate_left == 0) {
                if (lane == 0) mbar_arrive(&sm.gate);
                gate_left = -1;
            }
            stage = nstage;
            phase = nphase;
            ready = ready_next;
        }

        // ---- epilogue: one unsigned compare per accumulator against the row's threshold key ----
        // accumulator (mt, nt, e) of lane (g, q) is row 16w + mt*8 + perm(g), column nt*8 + perm(2q+e) = nt*8 + 4e + q.
        const long long pf_e0 = clock64();
        if (tr_on) tr[1] = pf_e0;
        if (lane < WROWS && shared_thr < w_thr[lane]) w_thr[lane] = shared_thr;
        if (SYM) cp_async_wait<0>();
        __syncwarp();
        u64* ck = a.cand_key + (size_t)seg * seg_stride;
        int* cj = a.cand_j + (size_t)seg * seg_stride;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            const int rw = mt * 8 + pg;                   // row within the warp's 16
            const u64 thr = w_thr[rw];
            unsigned mask = 0, cmask = 0;
#pragma unroll
            for (int nt = 0; nt < 16; ++nt) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const u64 bits = (u64)__double_as_longlong(acc[mt][nt][e]);
                    if (bits <= thr) mask |= 1u << (nt * 2 + e);
                    if (SYM && bits <= w_ct[nt * 8 + 4 * e + q4]) cmask |= 1u << (nt * 2 + e);
                }
            }
            if (mask | cmask) {
                // Rare path, kept deliberately compact (a fully unrolled version pushed the kernel far past the
                // instruction cache; a local-memory copy thrashed the tiny L1): park this row's 32 accumulators in
                // the warp's shared scratch, lane-interleaved, and walk the set bits.
                u64* tmp = w_sk + lane;                   // entry b lives at tmp[b * 32]
#pragma unroll
                for (int nt = 0; nt < 16; ++nt) {
                    tmp[(nt * 2) * 32] = (u64)__double_as_longlong(acc[mt][nt][0]);
                    tmp[(nt * 2 + 1) * 32] = (u64)__double_as_longlong(acc[mt][nt][1]);
                }
                const int cs = my_cs[mt];
                const unsigned clen = (unsigned)(my_ce[mt] - cs);
                unsigned m2 = mask;
                while (m2) {                               // drop inf / NaN scores and the row's own chromosome
                    const int bit = __ffs(m2) - 1;
                    m2 &= m2 - 1;
                    const int cl = (bit >> 1) * 8 + 4 * (bit & 1) + q4;
                    const unsigned hi32 = (unsigned)(tmp[bit * 32] >> 32);
                    if ((hi32 & 0x7ff00000u) == 0x7ff00000u || (unsigned)(col0 + cl - cs) < clen) mask &= ~(1u << bit);
                }
                if (mask) {                               // one shared-memory atomic per (thread, row)
                    pf_emit += __popc(mask);
                    int w = atomicAdd(&w_cnt[rw], __popc(mask));
                    u64* rk = ck + (size_t)(r0w + rw) * a.cap;
                    int* rj = cj + (size_t)(r0w + rw) * a.cap;
                    while (mask) {
                        const int bit = __ffs(mask) - 1;
                        mask &= mask - 1;
                        const int cl = (bit >> 1) * 8 + 4 * (bit & 1) + q4;
                        if (w < a.cap) {
                            rk[w] = tmp[bit * 32];
                            rj[w] = col0 + cl;
                        } else {
                            w_flag[rw] = 1;
                        }
                        ++w;
                    }
                }
                if (SYM && cmask) {
                    // column side: offer (bin j <- candidate i) to j's incoming buffer.  Rare (the thresholds are tight
                    // by the time the symmetric pass runs), so one global atomic per entry is affordable.
                    const int i = a.row_begin + rb * BM + r0w + rw;
                    while (cmask) {
                        const int bit = __ffs(cmask) - 1;
                        cmask &= cmask - 1;
                        const int j = col0 + (bit >> 1) * 8 + 4 * (bit & 1) + q4;
                        const u64 key = tmp[bit * 32];
                        if (((unsigned)(key >> 32) & 0x7ff00000u) == 0x7ff00000u || j >= a.N || i >= a.row_end) continue;
                        if ((unsigned)(j - cs) < clen) continue;     // same chromosome (i in j's range <=> j in i's range)
                        const int pos = atomicAdd(w_stgc, 1);
                        if (pos < STG) {
                            w_stg[pos] = make_uint4((unsigned)key, (unsigned)(key >> 32), (unsigned)j, (unsigned)i);
                        } else {                                     // staging full (loose thresholds): append directly
                            const int w = atomicAdd(a.in_cnt + j, 1);
                            if (w < a.in_cap) {
                                a.in_key[(size_t)j * a.in_cap + w] = key;
                                a.in_j[(size_t)j * a.in_cap + w] = i;
                            }
                        }
                        ++pf_emit;
                    }
                }
            }
        }
        __syncwarp();
        if (SYM && *w_stgc >= 32) flush_incoming();
        const long long pf_p0 = clock64();
        pf_epi += pf_p0 - pf_e0;
        if (tr_on) tr[2] = pf_p0;
        // ---- prune rows whose buffer could overflow during the next tile ----
        // (one ballot finds them: the common case - nothing to prune - costs a single shared-memory read per lane)
        prune_rows(__ballot_sync(0xffffffffu, lane < WROWS && w_cnt[lane] > a.cap - BN && !w_flag[lane]), ck, cj);
        pf_prune += clock64() - pf_p0;
        if (tr_on) tr[3] = clock64();
    }
    if (gate_left > 0 && lane == 0) mbar_arrive(&sm.gate);   // fewer chunks than the lag: open the gate on the way out
    __syncwarp();
    if (a.prof != nullptr && warp == 0 && lane == 0) {
        long long* o = a.prof + (size_t)blockIdx.x * 8;
        o[0] = clock64() - pf_t0; o[1] = pf_wait; o[2] = pf_epi; o[3] = pf_prune;
        o[4] = tcount; o[5] = pf_nprune; o[6] = pf_emit; o[7] = 0;
    }
}

#include "wc_search_f16.cuh"      // K4h / K5h: the same search with an fp16 tensor-core filter (option k5_f16 = 1, mma.sync)
#include "wc_search_tc.cuh"       // K5t: the fp16 filter on tcgen05 / TMEM (option k5_f16 = 2)

__global__ void wc_fill_u64_kernel(u64* p, size_t n, u64 v) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// ---------------------------------------------------------------------------------------------------------
// K4: centre at 1.0, row norms, the two extra samples; padding rows get (1, -inf) so they never pass the filter
// ---------------------------------------------------------------------------------------------------------
__global__ void wc_prepare_kernel(const double* __restrict__ X, int N, int Npad, int S, int ld, int Sx,
                                  double* __restrict__ Xc, double* __restrict__ norms) {
    const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= Npad) return;
    double* dst = Xc + (size_t)row * ld;
    double acc = 0.0;
    if (row < N) {
        const double* src = X + (size_t)row * S;
        for (int s = lane; s < ld; s += 32) {
            double v = s < S ? src[s] - 1.0 : 0.0;
            dst[s] = v;
            acc = fma(v, v, acc);
        }
    } else {
        for (int s = lane; s < ld; s += 32) dst[s] = 0.0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __syncwarp();
    if (lane == 0) {
        norms[row] = row < N ? acc : 0.0;
        dst[Sx] = 1.0;
        dst[Sx + 1] = row < N ? -0.5 * acc : -INFINITY;
    }
}

// ---------------------------------------------------------------------------------------------------------
// K6: per-row finalize
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool pair_less(double da, int ja, double db, int jb) {
    return da < db || (da == db && ja < jb);
}

struct FinArgs {
    const double* X;        // original corrected data, N x S
    int N, S;
    const double* norms;
    const int* row_cs;
    const int* row_ce;
    int row_begin, row_end;
    const int* rb_seg_first;
    const int* rb_seg_count;
    const u64* cand_key;
    const int* cand_j;
    const int* seg_cnt;
    const int* seg_flag;
    int cap;
    int k;
    int shortcap;           // shortlist capacity (256 or 512)
    double mcoef;
    int* idx_out;
    double* dist_out;
    int* slow_list;
    int* slow_count;
    int slow_bias;          // added to a row's number in slow_list (a call finalised in two row ranges: the second range's offset)
    int vec;                // 4: rows are 32-byte aligned (S % 4 == 0): 256-bit loads; 1: scalar loads
    const u64* in_key;      // symmetric search: the row's incoming (column-side) candidates, or nullptr
    const int* in_j;
    const int* in_cnt;
    int in_cap;
    double madd;            // window(v) = v + mcoef * (n_i + |v|) + madd
    const double* madd_p;   // when set: madd lives on the device
    const u64* row_thr;     // [rows] the tightest threshold key K5 published for the row (entries beyond it cannot rank), or nullptr
    int in_nsrc;            // incoming sources (1; one per rank after the exchange of a sharded symmetric search)
    int in_src_rows;        // rows between two sources: source s holds row r at (s * in_src_rows + r)
    // split form (select -> streaming re-score -> rank): the shortlist leaves the CTA
    int* sl_j;              // [rows][shortcap] shortlisted bins
    u64* sl_k;              // [rows][shortcap] their filter keys (histogram select only; the re-score's distance slots)
    int* sl_p;              // [rows] shortlist length; -1: the row is finished elsewhere (no candidates / exhaustive fallback)
    int* grp;               // work list of the re-score: (row << 4 | group of 32 shortlist slots)
    int* grp_count;
    const int* row_list;    // rows this launch handles (grid-stride), or nullptr: row = blockIdx.x
    const int* row_count;
    int* stats;             // split form: [0] live entries, [1] shortlisted candidates, [2] most live entries of a row; or nullptr
    // locality order of the re-score: a row's work items are filed under the smallest shortlisted bin (bucket = bin >> shift)
    int* sl_b;              // [rows] bucket of the row
    int* bkt_hist;          // [FIN_BUCKETS] work items per bucket
    int bkt_shift;
};

// One CTA per target row.
//  1. select: 256-bucket histogram over the row's candidate entries (all segments) -> v* = largest entry of the
//     bucket holding the k-th smallest approximate distance; shortlist = entries <= v* + margin(v*).  The
//     shortlist provably contains the exact top-k (every threshold ever applied to this row was >= that window).
//  2. exact re-score of the shortlist in the reference's operation order (wisetools.py:302 on Fortran-ordered
//     operands: sequential over samples, separately rounded subtract / multiply / add); one thread per
//     candidate, candidate rows staged through shared memory by cp.async in 32-sample chunks, double buffered.
//  3. rank by (distance, index), write the first k with indices remapped to other-chromosome coordinates.
// SPLIT: stop after step 1 and hand the shortlist to the streaming re-score (wc_fin_rescore_kernel) through global memory.
template <int FT, bool SPLIT>      // threads = shortlisted candidates re-scored per round: 128, or 160 behind the wider window of the fp16 filters
__device__ __forceinline__ void finalize_row(const FinArgs& a, const int rloc, unsigned char* fin_raw) {
    constexpr int ecap = FIN_ECAP;                                         // collected entries: [ecap] keys, [ecap] bins
    double* ex_d = reinterpret_cast<double*>(fin_raw + (size_t)ecap * 12); // shortcap
    int* ex_j = reinterpret_cast<int*>(ex_d + a.shortcap);                 // shortcap
    int* hist = ex_j + a.shortcap;                                         // HIST_BINS
    __shared__ double s_red[2][FT / 32];
    __shared__ int s_total, s_flag, s_p, s_bstar, s_valid;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int row = a.row_begin + rloc;
    const int rb = rloc / BM, rl = rloc % BM;
    const int seg0 = a.rb_seg_first[rb], nseg = a.rb_seg_count[rb];
    int* out_i = a.idx_out + (size_t)rloc * a.k;
    double* out_d = a.dist_out + (size_t)rloc * a.k;

    // candidate sources of the row: its segments (one per K5 piece of the row block and column half) and, after a symmetric
    // search, the incoming buffer(s)
    const int nsrc = nseg + (a.in_key != nullptr ? a.in_nsrc : 0);
    auto source = [&](int s, const u64*& keys, const int*& js, int& flagged) -> int {
        if (s < nseg) {
            const size_t off = ((size_t)(seg0 + s) * BM + rl) * a.cap;
            keys = a.cand_key + off;
            js = a.cand_j + off;
            flagged = a.seg_flag[(size_t)(seg0 + s) * BM + rl];
            return a.seg_cnt[(size_t)(seg0 + s) * BM + rl];
        }
        const size_t r = (size_t)(s - nseg) * a.in_src_rows + rloc;
        keys = a.in_key + r * a.in_cap;
        js = a.in_j + r * a.in_cap;
        const int n = a.in_cnt[r];
        flagged = n > a.in_cap ? 1 : 0;               // more offers than the buffer holds: exact fallback
        return n < a.in_cap ? n : a.in_cap;
    };
    // ---- 0. collect: every warp walks its share of the sources, the row's entries land side by side in shared memory (the
    //         staging tiles are idle until the re-score) - the select passes below never touch global memory again ----
    u64* en_k = reinterpret_cast<u64*>(fin_raw);                                     // [ecap]
    int* en_j = reinterpret_cast<int*>(en_k + ecap);                                 // [ecap]
    if (tid == 0) { s_total = 0; s_flag = 0; s_p = 0; s_valid = 0; }
    for (int b = tid; b < HIST_BINS; b += FT) hist[b] = 0;
    const u64 tfinal = a.row_thr != nullptr ? __ldcg(a.row_thr + rloc) : ~0ull;
    __syncthreads();
    for (int s = warp; s < nsrc; s += FT / 32) {
        const u64* cd;
        const int* cjs;
        int fl;
        const int n = source(s, cd, cjs, fl);
        if (fl) { if (lane == 0) s_flag = 1; continue; }
        for (int e0 = 0; e0 < n; e0 += 32) {
            const int e = e0 + lane;
            // Entries beyond the row's final threshold are dead weight: every published threshold is (k-th smallest filter
            // distance of a SUBSET of the candidates) + margin, hence >= the window the shortlist is cut at below.
            const u64 key = e < n ? cd[e] : ~0ull;
            const bool keep = e < n && key <= tfinal;
            const unsigned bm = __ballot_sync(0xffffffffu, keep);
            if (bm == 0u) continue;
            int base = 0;
            if (lane == 0) base = atomicAdd(&s_total, __popc(bm));
            base = __shfl_sync(0xffffffffu, base, 0) + __popc(bm & ((1u << lane) - 1u));
            if (keep && base < ecap) {
                en_k[base] = key;
                en_j[base] = cjs[e];
            }
        }
    }
    __syncthreads();
    const int total = s_total;
    if (s_flag) {
        if (tid == 0) {
            a.slow_list[atomicAdd(a.slow_count, 1)] = rloc + a.slow_bias;
            if (SPLIT) a.sl_p[rloc] = -1;
        }
        return;
    }
    if (total == 0) {
        for (int e = tid; e < a.k; e += FT) { out_i[e] = -1; out_d[e] = 1e10; }
        if (SPLIT && tid == 0) a.sl_p[rloc] = -1;
        return;
    }
    // The select passes visit every live entry of the row: from shared memory when the collection fitted (the normal case),
    // else straight from the sources (rows no segment ever pruned: small matrices).
    const bool in_smem = total <= ecap;
    auto for_each_entry = [&](auto&& f) {
        if (in_smem) {
            for (int e = tid; e < total; e += FT) f(en_k[e], en_j[e]);
        } else {
            for (int s2 = 0; s2 < nsrc; ++s2) {
                const u64* cd;
                const int* cjs;
                int fl;
                const int n = source(s2, cd, cjs, fl);
                for (int e = tid; e < n; e += FT) {
                    const u64 key = cd[e];
                    if (key <= tfinal) f(key, cjs[e]);
                }
            }
        }
    };

    // ---- 1. select ----
    double mn = INFINITY, mx = -INFINITY;
    for_each_entry([&](u64 key, int) {
        const double d = dist_of_key(key);
        mn = fmin(mn, d);
        mx = fmax(mx, d);
    });
    mn = warp_min(mn);
    mx = warp_max(mx);
    if (lane == 0) { s_red[0][warp] = mn; s_red[1][warp] = mx; }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < FT / 32; ++w) { mn = fmin(mn, s_red[0][w]); mx = fmax(mx, s_red[1][w]); }
    const float scale = (mx > mn) ? (float)(HIST_BINS - 1) / (float)(mx - mn) : 0.0f;
    for_each_entry([&](u64 key, int) { atomicAdd(&hist[bucket_of(dist_of_key(key), mn, scale)], 1); });
    __syncthreads();
    if (warp == 0) {
        int c[HIST_BINS / 32], sum = 0;
#pragma unroll
        for (int t = 0; t < HIST_BINS / 32; ++t) { c[t] = hist[lane * (HIST_BINS / 32) + t]; sum += c[t]; }
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        int run = incl - sum, bl = -1;
#pragma unroll
        for (int t = 0; t < HIST_BINS / 32; ++t) {
            run += c[t];
            if (bl < 0 && run >= a.k) bl = lane * (HIST_BINS / 32) + t;
        }
        unsigned m = __ballot_sync(0xffffffffu, bl >= 0);
        int bstar = HIST_BINS - 1;                      // fewer than k entries: keep them all
        if (m) bstar = __shfl_sync(0xffffffffu, bl, __ffs(m) - 1);
        if (lane == 0) s_bstar = bstar;
    }
    __syncthreads();
    const int bstar = s_bstar;
    double vstar = -INFINITY;
    for_each_entry([&](u64 key, int) {
        const double d = dist_of_key(key);
        if (bucket_of(d, mn, scale) <= bstar) vstar = fmax(vstar, d);
    });
    vstar = warp_max(vstar);
    __syncthreads();                                    // s_red reuse
    if (lane == 0) s_red[0][warp] = vstar;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < FT / 32; ++w) vstar = fmax(vstar, s_red[0][w]);
    const double window = vstar + a.mcoef * (a.norms[row] + fabs(vstar)) + madd_of(a);
    for_each_entry([&](u64 key, int j) {
        if (dist_of_key(key) <= window) {
            const int slot = atomicAdd(&s_p, 1);
            if (slot < a.shortcap) ex_j[slot] = j;
        }
    });
    __syncthreads();
    const int p = s_p;
    if (p > a.shortcap) {                               // tie plateau wider than the shortlist: exact fallback
        if (tid == 0) {
            a.slow_list[atomicAdd(a.slow_count, 1)] = rloc + a.slow_bias;
            if (SPLIT) a.sl_p[rloc] = -1;
        }
        return;
    }
    if (SPLIT) {                                        // the shortlist goes to the streaming re-score, 32 slots per work item
        for (int e = tid; e < p; e += FT) a.sl_j[(size_t)rloc * a.shortcap + e] = ex_j[e];
        if (tid == 0) {
            a.sl_p[rloc] = p;
            const int ng = (p + 31) >> 5;
            int jmin = 0x7fffffff;
            for (int e = 0; e < p; ++e) jmin = min(jmin, ex_j[e]);
            const int bkt = min(jmin >> a.bkt_shift, FIN_BUCKETS - 1);
            a.sl_b[rloc] = bkt;
            atomicAdd(a.bkt_hist + bkt, ng);
            if (a.stats != nullptr) { atomicAdd(a.stats, total); atomicAdd(a.stats + 1, p); }
        }
        return;
    }

    // ---- 2. exact re-score ----
    // (Tried and dropped, r02u/v: four lanes fetching one whole 128-byte line per load with a swizzled warp-private shared-memory
    // patch transposing it back - the L2 request count fell 4x (lts 53 % -> 23 %) but the extra shared-memory wavefronts and the
    // lost occupancy cost more: 6.5 / 9.0 ms against 6.2 ms.)
    // One thread per shortlisted candidate.  The candidate's row streams from L2 straight into registers - eight 256-bit
    // loads (32 samples) in flight per thread, nothing staged, no barrier inside the loop - while the target's own row is a
    // broadcast operand in shared memory.  The sum runs strictly in sample order with separately rounded subtract, multiply
    // and add (wisetools.py:302 on Fortran-ordered operands).
    const double* xrow = a.X + (size_t)row * a.S;
    double* xi_s = reinterpret_cast<double*>(fin_raw);          // the collected entries are dead: the area now holds the row
    const bool xi_in_smem = (size_t)a.S * 8 <= (size_t)ecap * 12;
    __syncthreads();
    if (xi_in_smem)
        for (int t = tid; t < a.S; t += FT) xi_s[t] = xrow[t];
    __syncthreads();
    const uint32_t xi_u32 = smem_u32(xi_s);
    for (int c0 = 0; c0 < p; c0 += FT) {
        if (c0 + warp * 32 < p) {                                // warp-uniform; idle lanes shadow the last candidate
            const bool live = c0 + tid < p;
            const int j = ex_j[live ? c0 + tid : p - 1];
            const double* xr = a.X + (size_t)j * a.S;
            double accd = 0.0;
            int t0 = 0;
            if (a.vec == 4 && xi_in_smem) {
                for (; t0 + 32 <= a.S; t0 += 32) {
                    double v[32];
#pragma unroll
                    for (int u = 0; u < 8; ++u) ldg_nc_v4f64(xr + t0 + 4 * u, v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]);
                    // ptxas would sink the loads between the dependent adds (three in flight, 96 contiguous bytes); memory
                    // operations do not move across a warp barrier, so all eight are issued here: 256 contiguous bytes per lane
                    __syncwarp();
#pragma unroll
                    for (int u = 0; u < 16; ++u) {
                        double x0, x1;
                        lds_v2f64(xi_u32 + (uint32_t)(t0 + 2 * u) * 8u, x0, x1);
                        double d = __dsub_rn(v[2 * u], x0);
                        accd = __dadd_rn(accd, __dmul_rn(d, d));
                        d = __dsub_rn(v[2 * u + 1], x1);
                        accd = __dadd_rn(accd, __dmul_rn(d, d));
                    }
                }
                for (; t0 + 4 <= a.S; t0 += 4) {
                    double v0, v1, v2, v3;
                    ldg_nc_v4f64(xr + t0, v0, v1, v2, v3);
                    double d = __dsub_rn(v0, xi_s[t0]);     accd = __dadd_rn(accd, __dmul_rn(d, d));
                    d = __dsub_rn(v1, xi_s[t0 + 1]);        accd = __dadd_rn(accd, __dmul_rn(d, d));
                    d = __dsub_rn(v2, xi_s[t0 + 2]);        accd = __dadd_rn(accd, __dmul_rn(d, d));
                    d = __dsub_rn(v3, xi_s[t0 + 3]);        accd = __dadd_rn(accd, __dmul_rn(d, d));
                }
            }
            if (xi_in_smem) {
                for (; t0 < a.S; ++t0) {
                    const double d = __dsub_rn(__ldg(xr + t0), xi_s[t0]);
                    accd = __dadd_rn(accd, __dmul_rn(d, d));
                }
            } else {                                             // more samples than the area holds: both rows from global memory
                for (; t0 < a.S; ++t0) {
                    const double d = __dsub_rn(__ldg(xr + t0), __ldg(xrow + t0));
                    accd = __dadd_rn(accd, __dmul_rn(d, d));
                }
            }
            __syncwarp();                    // every lane has read its candidate's bin before the live lanes overwrite theirs
            if (live) {
                const bool ok = accd < 1e10;     // wisetools.py:312-314: strict `<` against the 1e10 start value; NaN fails
                ex_d[c0 + tid] = ok ? accd : INFINITY;
                ex_j[c0 + tid] = ok ? j : 0x7fffffff;
            }
        }
    }
    __syncthreads();

    // ---- 3. rank by (distance, index) and write ----
    const int cs = a.row_cs[row], ce = a.row_ce[row];
    int nvalid_local = 0;
    for (int e = tid; e < p; e += FT) {
        const double d = ex_d[e];
        const int j = ex_j[e];
        if (j == 0x7fffffff) continue;
        ++nvalid_local;
        int rank = 0;
        for (int u = 0; u < p; ++u) rank += pair_less(ex_d[u], ex_j[u], d, j) ? 1 : 0;
        if (rank < a.k) {
            out_i[rank] = j >= ce ? j - (ce - cs) : j;
            out_d[rank] = d;
        }
    }
    atomicAdd(&s_valid, nvalid_local);
    __syncthreads();
    for (int e = s_valid + tid; e < a.k; e += FT) { out_i[e] = -1; out_d[e] = 1e10; }
}

// One CTA per target row (grid = rows), or - with a row list (the rows the warp-per-row select of the split form passed on:
// more live entries than a warp holds) - a fixed grid striding over the list.
template <int FT, bool SPLIT>
__global__ void __launch_bounds__(FT) wc_finalize_kernel(const FinArgs a) {
    extern __shared__ __align__(32) unsigned char fin_raw[];
    if (a.row_list == nullptr) {
        finalize_row<FT, SPLIT>(a, (int)blockIdx.x, fin_raw);
        return;
    }
    const int n = *a.row_count;
    for (int b = blockIdx.x; b < n; b += gridDim.x) {
        finalize_row<FT, SPLIT>(a, a.row_list[b], fin_raw);
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------
// K6b: exhaustive exact search for one row per CTA (rare)
// ---------------------------------------------------------------------------------------------------------
struct ExhArgs {
    const double* X;
    int N, S;
    const int* row_cs;
    const int* row_ce;
    int row_begin;
    const int* slow_list;
    int list_off;
    double* scratch;     // [rows in this batch][N]
    int k;
    int* idx_out;
    double* dist_out;
};

__global__ void __launch_bounds__(EXH_THREADS) wc_exhaustive_kernel(const ExhArgs a) {
    __shared__ double s_d[EXH_THREADS / 32];
    __shared__ int s_j[EXH_THREADS / 32];
    __shared__ double s_bd;
    __shared__ int s_bj;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rloc = a.slow_list[a.list_off + blockIdx.x];
    const int row = a.row_begin + rloc;
    const int cs = a.row_cs[row], ce = a.row_ce[row];
    double* dd = a.scratch + (size_t)blockIdx.x * a.N;
    const double* xrow = a.X + (size_t)row * a.S;
    for (int j = tid; j < a.N; j += EXH_THREADS) {
        double acc = INFINITY;
        if (j < cs || j >= ce) {
            const double* xj = a.X + (size_t)j * a.S;
            acc = 0.0;
            for (int s = 0; s < a.S; ++s) {
                double v = __dsub_rn(xj[s], xrow[s]);
                acc = __dadd_rn(acc, __dmul_rn(v, v));
            }
            if (!(acc < 1e10)) acc = INFINITY;
        }
        dd[j] = acc;
    }
    __syncthreads();
    double last_d = -INFINITY;
    int last_j = -1;
    int* out_i = a.idx_out + (size_t)rloc * a.k;
    double* out_d = a.dist_out + (size_t)rloc * a.k;
    for (int t = 0; t < a.k; ++t) {
        double bd = INFINITY;
        int bj = 0x7fffffff;
        for (int j = tid; j < a.N; j += EXH_THREADS) {
            double d = dd[j];
            bool after = d > last_d || (d == last_d && j > last_j);
            if (after && pair_less(d, j, bd, bj)) { bd = d; bj = j; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double od = __shfl_xor_sync(0xffffffffu, bd, o);
            int oj = __shfl_xor_sync(0xffffffffu, bj, o);
            if (pair_less(od, oj, bd, bj)) { bd = od; bj = oj; }
        }
        if (lane == 0) { s_d[warp] = bd; s_j[warp] = bj; }
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < EXH_THREADS / 32; ++w)
                if (pair_less(s_d[w], s_j[w], bd, bj)) { bd = s_d[w]; bj = s_j[w]; }
            s_bd = bd;
            s_bj = bj;
            if (bd < INFINITY) {
                out_i[t] = bj >= ce ? bj - (ce - cs) : bj;
                out_d[t] = bd;
            } else {
                out_i[t] = -1;
                out_d[t] = 1e10;
            }
        }
        __syncthreads();
        last_d = s_bd;
        last_j = s_bj;
        if (!(last_d < INFINITY)) {          // everything left is a filler
            for (int e = t + 1 + tid; e < a.k; e += EXH_THREADS) { out_i[e] = -1; out_d[e] = 1e10; }
            break;
        }
    }
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

namespace {
// Which CTA computes which tiles, in which order.  prefix[rb+1]-prefix[rb] = number of tiles of row block rb; a piece
// is (row block, arithmetic progression q0, q0+step, ... < q1 over that block's tile indices).
// The centred matrix (Npad x ld doubles; 288 MB at 600 x 50 kb) does not fit the 126 MB L2, and every tile needs a
// 128-row A panel and a 128-row B panel of it.  With CTAs spread over unrelated columns every panel comes from DRAM for
// every tile (measured: 188 GB per launch at 600 x 50 kb).  So work is handed out in *rounds*: in a round a group of G
// CTAs shares one row block and walks its tiles interleaved (CTA j takes tiles j, j+G, ...), all groups starting
// together.  The CTAs then sit on (nearly) the same B panel at the same time - it is read from DRAM once per round -
// and the live A panels (grid/G of them) stay L2-resident.  Row blocks left after the last full round are cut into
// contiguous ranges that level the CTAs' tile counts (water-filling), so the balance of the plain equal split is kept.
#include "wc_search_fin.cuh"      // K6 split form: streaming re-score + rank, and the K6 launch shared by both search entries
#include "wc_search_wide.cuh"     // K5w / K6w: the wide-refsize search (wc_newref_topk_wide)

struct Piece { int cta, rb, q0, q1, step, seg, pass; };
void schedule_pieces(const std::vector<int>& prefix, int nrb, int grid, int G, bool rounds_on, int pass,
                     std::vector<Piece>& pieces) {
    std::vector<long long> load(grid, 0);
    if (G > grid) G = grid;
    if (G < 1) G = 1;
    const int groups = grid / G;
    const int rounds = rounds_on ? nrb / groups : 0;
    for (int r = 0; r < rounds; ++r)
        for (int g = 0; g < groups; ++g) {
            const int rb = r * groups + g;
            const int nv = prefix[rb + 1] - prefix[rb];
            for (int j = 0; j < G && j < nv; ++j) {
                pieces.push_back({g * G + j, rb, j, nv, G, 0, pass});
                load[g * G + j] += (nv - j + G - 1) / G;
            }
        }
    const int rb_left = rounds * groups;
    long long left = prefix[nrb] - prefix[rb_left];
    if (left > 0) {
        long long lo = 0, hi = 0;
        for (int c = 0; c < grid; ++c) hi = std::max(hi, load[c]);
        hi += left;                                       // level with sum(max(0, level - load)) >= left
        while (lo < hi) {
            const long long mid = (lo + hi) / 2;
            long long cap_sum = 0;
            for (int c = 0; c < grid; ++c) cap_sum += std::max(0ll, mid - load[c]);
            if (cap_sum >= left) hi = mid; else lo = mid + 1;
        }
        int rb = rb_left, q = 0;
        for (int c = 0; c < grid && left > 0; ++c) {
            long long want = std::min(left, std::max(0ll, lo - load[c]));
            while (want > 0) {
                const int nv = prefix[rb + 1] - prefix[rb];
                if (q >= nv) { ++rb; q = 0; continue; }
                const int take = (int)std::min<long long>(want, nv - q);
                pieces.push_back({c, rb, q, q + take, 1, 0, pass});
                load[c] += take;
                q += take;
                want -= take;
                left -= take;
            }
        }
    }
}

// Symmetric search: which column tiles each block of 128 bins computes.  skip_lo / skip_n: per block the column tiles
// wholly inside its own chromosome.  Pass A (list_a): the symmetric subset (I + J) % frac == 0 and the diagonal, from
// both sides.  Pass B (list_b): every other pair once - block I takes J = I + 1 ... I + nb/2 cyclically, the antipodal
// pair of an even nb belongs to its lower block.  Lists are built for the blocks [b0, b1) (a rank's share), off_* are
// relative to b0.  tools: wc_debug_sym_plan exposes this to the CPU tests (coverage: every needed pair exactly once).
void pair_lists(int nb, const std::vector<int>& skip_lo, const std::vector<int>& skip_n, int frac, int b0, int b1,
                std::vector<int>& list_a, std::vector<int>& off_a, std::vector<int>& list_b, std::vector<int>& off_b) {
    auto in_sample = [&](int I, int J) { return I == J || (I + J) % frac == 0; };
    auto valid = [&](int I, int t) { return !(t >= skip_lo[I] && t < skip_lo[I] + skip_n[I]); };
    list_a.clear();
    list_b.clear();
    off_a.assign(b1 - b0 + 1, 0);
    off_b.assign(b1 - b0 + 1, 0);
    for (int I = b0; I < b1; ++I) {
        for (int t = 0; t < nb; ++t)
            if (valid(I, t) && in_sample(I, t)) list_a.push_back(t);
        off_a[I - b0 + 1] = (int)list_a.size();
        for (int dlt = 1; dlt <= nb / 2; ++dlt) {
            if (2 * dlt == nb && I >= nb / 2) continue;
            const int t = (I + dlt) % nb;
            if (valid(I, t) && !in_sample(I, t)) list_b.push_back(t);
        }
        off_b[I - b0 + 1] = (int)list_b.size();
    }
}

// Exclusion range [cs, ce) of every bin (its own chromosome) and the skipped column tiles of every whole-matrix block.
void block_skips(int N, const int* chrom_bins_h, int nchrom, std::vector<int>& row_cs, std::vector<int>& row_ce,
                 std::vector<int>& skip_lo, std::vector<int>& skip_n) {
    row_cs.assign(N, 0);
    row_ce.assign(N, 0);
    int pos = 0;
    for (int c = 0; c < nchrom; ++c) {
        for (int i = 0; i < chrom_bins_h[c]; ++i) { row_cs[pos + i] = pos; row_ce[pos + i] = pos + chrom_bins_h[c]; }
        pos += chrom_bins_h[c];
    }
    const int nb = (N + BM - 1) / BM;
    skip_lo.assign(nb, nb);
    skip_n.assign(nb, 0);
    for (int I = 0; I < nb; ++I) {
        const int r0 = I * BM, r1 = std::min(N, r0 + BM) - 1;
        if (row_cs[r0] == row_cs[r1]) {   // block inside one chromosome: its interior column tiles are skipped
            const int first = (row_cs[r0] + BN - 1) / BN, last = row_ce[r0] / BN;
            if (last > first) { skip_lo[I] = first; skip_n[I] = last - first; }
        }
    }
}

}  // namespace


namespace {
// Tensor map of a row-major fp16 matrix [rows][ldh] with boxes of 64 halves x 128 rows, SWIZZLE_128B (the operand tiles of
// K5h / K5t).
int encode_f16_map(wc_ctx* ctx, CUtensorMap* tmap, const void* base, int ldh, size_t rows) {      // ldh: row width = row stride, in halves
    if (!ctx->encode_tiled) {
        wc_set_error("cuTensorMapEncodeTiled is not available from this driver");
        return WC_ERR_CUDA;
    }
    cuuint64_t dims[2] = {(cuuint64_t)ldh, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ldh * sizeof(__half)};
    cuuint32_t box[2] = {(cuuint32_t)BKH, BM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = reinterpret_cast<PFN_encodeTiled>(ctx->encode_tiled)(
        tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        wc_set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
        return WC_ERR_CUDA;
    }
    return WC_OK;
}

// Pivots of a search over N bins with refsize k: TC_PIVOTS (their distances to 128 bins fill the tensor memory), or 0 - no
// pivot pass - when the matrix is too small for it to pay or refsize leaves too few pivots per bin.
int pivot_count(int N, int k) {
    return (k <= 128 && (long long)TC_PIVOTS * 4 <= N) ? TC_PIVOTS : 0;
}

// The pivot pass of K5t (see wc_search_tc.cuh): thresholds of the target bins of row blocks [0, nrb) (relative to
// ta.row_begin) from their distances to the R bins of smallest norm.  `ta` arrives prepared for the search proper (norms,
// exclusion ranges, candidate buffers, margins, row_thr, n32); rb_seg_first[rb] names a segment of row block rb whose
// candidate buffers serve as scratch - the search proper overwrites them afterwards.
int tc_pivot_pass(wc_ctx* ctx, cudaStream_t stream, const CUtensorMap& tmap_a, TopkArgs ta, const __half* Xh, int ldh, int ldx, int N,
                  int nrb, const std::vector<int>& rb_seg_first, int R) {
    int* ids; __half* P; float* n32p; int* meta;
    int rc;
    if ((rc = wc_reserve(ctx, SLOT_PIV_IDS, (size_t)R * sizeof(int), (void**)&ids))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_PIV_X, (size_t)R * ldh * sizeof(__half), (void**)&P))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_PIV_N, (size_t)R * sizeof(float), (void**)&n32p))) return rc;
    if (R != TC_PIVOTS) { wc_set_error("pivot pass: %d pivots unsupported", R); return WC_ERR_INTERNAL; }
    const int gridP = std::max(1, std::min(ctx->sm_count, nrb));
    std::vector<int> m((size_t)gridP + 1 + (size_t)nrb * 5);
    {
        int w = 0;
        for (int c = 0; c < gridP; ++c) {
            m[c] = w;
            for (int rb = c; rb < nrb; rb += gridP, ++w) {
                int* pc = &m[(size_t)gridP + 1 + (size_t)w * 5];
                pc[0] = rb; pc[1] = 0; pc[2] = R / BN; pc[3] = 1; pc[4] = rb_seg_first[rb];
            }
        }
        m[gridP] = w;
    }
    if ((rc = wc_reserve(ctx, SLOT_PIV_META, m.size() * sizeof(int), (void**)&meta))) return rc;
    unsigned long long h = 1469598103934665603ull;
    for (int v : m) { h ^= (unsigned)v; h *= 1099511628211ull; }
    h ^= (unsigned long long)(uintptr_t)meta;
    if (h != ctx->piv_hash) {
        WC_CUDA(cudaMemcpyAsync(meta, m.data(), m.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
        ctx->piv_hash = h;
    }
    wc_pivot_select_kernel<<<1, 1024, 0, stream>>>(ta.n32, N, R, ids);
    wc_pivot_gather_kernel<<<R, 128, 0, stream>>>(Xh, ldh, ldx, ta.n32, ids, P, n32p);
    WC_CUDA(cudaGetLastError());
    CUtensorMap tmap_p;
    if ((rc = encode_f16_map(ctx, &tmap_p, P, ldh, (size_t)R))) return rc;
    ta.cta_piece_begin = meta; ta.pieces = meta + gridP + 1;
    ta.tile_list = nullptr; ta.rb_list_off = nullptr; ta.final_prune = 1;
    ta.in_key = nullptr; ta.in_j = nullptr; ta.in_cnt = nullptr; ta.in_cap = 0; ta.col_thr = nullptr;
    ta.coln32 = n32p; ta.col_ids = ids; ta.dbg = nullptr; ta.dbg_ld = 0; ta.prof = nullptr; ta.trace = nullptr;
    ta.kb_last = ldh - BKH;               // the pivot matrix carries the B version of the last chunk in place
    WC_CUDA(cudaFuncSetAttribute(wc_dist_topk_tc_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_BYTES));
    wc_dist_topk_tc_kernel<2, false><<<gridP, TC_THREADS, TC_SMEM_BYTES, stream>>>(tmap_a, tmap_p, ta);
    WC_CUDA(cudaGetLastError());
    return WC_OK;
}
}  // namespace

// CPU-only debug aid (no device, no context): the symmetric search's tile lists and CTA schedule for the blocks of rank
// `rank` of `world`.  out: [nb, b0, b1, nA, nB, piecesA, piecesB, 0][off_a nrb+1][off_b nrb+1][list_a][list_b]
// [pieces of pass A: cta, row block, q0, q1, step]...[pieces of pass B]...[skip_lo nb][skip_n nb].
extern "C" int wc_debug_sym_plan(int N, const int* chrom_bins_h, int nchrom, int frac, int world, int rank, int grid,
                                 int group, int rounds_on, int* out, long long out_ints, long long* used) {
    WC_CHECK_ARG(N > 0 && chrom_bins_h != nullptr && nchrom > 0 && frac >= 2 && world >= 1 && rank >= 0 && rank < world);
    WC_CHECK_ARG(grid >= 1 && group >= 1 && out != nullptr && used != nullptr);
    long long tot = 0;
    for (int c = 0; c < nchrom; ++c) { WC_CHECK_ARG(chrom_bins_h[c] >= 0); tot += chrom_bins_h[c]; }
    WC_CHECK_ARG(tot == N);
    std::vector<int> row_cs, row_ce, skip_lo, skip_n, la, oa, lb, ob;
    block_skips(N, chrom_bins_h, nchrom, row_cs, row_ce, skip_lo, skip_n);
    const int nb = (N + BM - 1) / BM;
    const int bp = (nb + world - 1) / world;
    const int b0 = std::min(nb, rank * bp), b1 = std::min(nb, b0 + bp), nrb = b1 - b0;
    pair_lists(nb, skip_lo, skip_n, frac, b0, b1, la, oa, lb, ob);
    std::vector<Piece> pa, pb;
    if (!la.empty()) schedule_pieces(oa, nrb, std::max(1, std::min<int>(grid, ((int)la.size() + 7) / 8)), 1, false, 0, pa);
    if (!lb.empty()) schedule_pieces(ob, nrb, std::max(1, std::min<int>(grid, ((int)lb.size() + 7) / 8)), group, rounds_on != 0, 1, pb);
    const long long need = 8 + 2ll * (nrb + 1) + (long long)la.size() + (long long)lb.size() + 5ll * (pa.size() + pb.size()) + 2ll * nb;
    *used = need;
    if (need > out_ints) { wc_set_error("wc_debug_sym_plan: %lld ints needed", need); return WC_ERR_ARG; }
    int* o = out;
    *o++ = nb; *o++ = b0; *o++ = b1; *o++ = (int)la.size(); *o++ = (int)lb.size(); *o++ = (int)pa.size(); *o++ = (int)pb.size(); *o++ = 0;
    for (int v : oa) *o++ = v;
    for (int v : ob) *o++ = v;
    for (int v : la) *o++ = v;
    for (int v : lb) *o++ = v;
    for (const std::vector<Piece>* pv : {&pa, &pb})
        for (const Piece& pc : *pv) { *o++ = pc.cta; *o++ = pc.rb; *o++ = pc.q0; *o++ = pc.q1; *o++ = pc.step; }
    for (int v : skip_lo) *o++ = v;
    for (int v : skip_n) *o++ = v;
    return WC_OK;
}

namespace {
// madd of the fp16 filter from K4h's statistics (stats[0] = bits of the largest norm): out = 2 eps nmax + 2^-20 sqrt(S nmax)
__global__ void wc_f16_margin_kernel(const unsigned long long* __restrict__ stats, int S, double eps16, double* __restrict__ out) {
    const double nmax = __longlong_as_double((long long)stats[0]);
    out[0] = 2.0 * eps16 * nmax + ldexp(1.0, -20) * sqrt((double)S * nmax);
}
}  // namespace

namespace {
// Host plan of a search (see wc_newref_topk), cached in the context between identical calls.
struct SearchPlan {
    unsigned long long key = 0, content_hash = 0;
    bool valid = false;
    std::vector<int> row_cs, row_ce, skip_lo, skip_n, rb_seg_first, rb_seg_count, cta_piece_begin, piece_tab, sym_tab;
    int nrb = 0, total_tiles = 0, grid = 0, sym = 0, sym_frac = 0, gridA = 0, gridB = 0, grid0 = 0, nseg = 0;
    long long tilesA = 0, tilesB = 0;
    size_t listA_size = 0;
};
}  // namespace

extern "C" int wc_newref_topk(wc_ctx* ctx, const double* corrected_d, int N, int S, const int* chrom_bins_h,
                              int nchrom, int row_begin, int row_end, int refsize, int32_t* idx_d, double* dist_d,
                              void* stream_v) {
    WC_CHECK_ARG(ctx != nullptr);
    WC_CHECK_ARG(corrected_d != nullptr && chrom_bins_h != nullptr);
    WC_CHECK_ARG(N > 0 && S > 0 && nchrom > 0);
    WC_CHECK_ARG(refsize >= 1 && refsize <= 384);
    WC_CHECK_ARG(row_begin >= 0 && row_begin <= row_end && row_end <= N);
    long long tot = 0;
    for (int c = 0; c < nchrom; ++c) {
        WC_CHECK_ARG(chrom_bins_h[c] >= 0);
        tot += chrom_bins_h[c];
    }
    WC_CHECK_ARG(tot == N);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    WC_CUDA(cudaSetDevice(ctx->device));
    for (int i = 0; i < 4; ++i) ctx->phase_ms[i] = 0.0;
    for (int i = 0; i < 5; ++i) ctx->counter[i] = 0;
    ctx->timed_mask &= ~0xfu;
    const int rows = row_end - row_begin;
    if (rows == 0) return WC_OK;
    WC_CHECK_ARG(idx_d != nullptr && dist_d != nullptr);

    const int k = refsize;
    const int cap = k <= 128 ? 512 : 1024;
    // sample axis: nblocks 8-sample blocks of data, then one block holding the two extra samples (1, -n/2)
    const int nblocks = (S + 7) / 8;
    const int Sx = nblocks * 8;
    const int nkc = nblocks / 2 + 1;
    const int nd_last = nblocks - 2 * (nkc - 1);          // 0 or 1 data double-steps in the last chunk
    const int extra_h = nd_last;
    const int ld = nkc * BK;
    const size_t Npad = (size_t)(N + BN - 1) / BN * BN + BN;
    const double mcoef = 16.0 * (double)(S + 16) * 1.1102230246251565e-16;

    // ---- host plan: exclusion ranges, work list, schedule.  A pure function of (N, chromosome sizes, row range, refsize, SM
    //      count, options): repeated calls on the same problem (bench loops, the parts of one newref) reuse it - building it
    //      costs ~0.5 ms of host time at 50 kb during which the GPU would idle ----
    unsigned long long plan_key = 1469598103934665603ull;
    {
        auto mixk = [&](const void* p, size_t bytes) {
            const unsigned char* c = static_cast<const unsigned char*>(p);
            for (size_t i = 0; i < bytes; ++i) { plan_key ^= c[i]; plan_key *= 1099511628211ull; }
        };
        mixk(chrom_bins_h, (size_t)nchrom * sizeof(int));
        const int dims[10] = {N, nchrom, row_begin, row_end, refsize, ctx->sm_count, ctx->k5_sym, ctx->k5_group, ctx->k5_f16, 0x5ea7c4};
        mixk(dims, sizeof(dims));
    }
    if (ctx->search_plan == nullptr) {
        ctx->search_plan = new SearchPlan();
        ctx->search_plan_free = [](void* q) { delete static_cast<SearchPlan*>(q); };
    }
    SearchPlan& P = *static_cast<SearchPlan*>(ctx->search_plan);
    if (P.key != plan_key || !P.valid) {
    P.valid = false;
    std::vector<int> row_cs(N), row_ce(N);
    {
        int pos = 0;
        for (int c = 0; c < nchrom; ++c) {
            for (int i = 0; i < chrom_bins_h[c]; ++i) {
                row_cs[pos + i] = pos;
                row_ce[pos + i] = pos + chrom_bins_h[c];
            }
            pos += chrom_bins_h[c];
        }
    }
    const int nrb = (rows + BM - 1) / BM;
    const int ntile_cols = (N + BN - 1) / BN;
    std::vector<int> prefix(nrb + 1), skip_lo(nrb), skip_n(nrb);
    prefix[0] = 0;
    for (int rb = 0; rb < nrb; ++rb) {
        int r0 = row_begin + rb * BM;
        int r1 = std::min(row_end, r0 + BM) - 1;
        int lo = ntile_cols, n = 0;
        if (row_cs[r0] == row_cs[r1]) {   // block inside one chromosome: its interior column tiles are skipped
            int first = (row_cs[r0] + BN - 1) / BN;
            int last = row_ce[r0] / BN;    // tiles [first, last) lie wholly inside [cs, ce)
            if (last > first) { lo = first; n = last - first; }
        }
        skip_lo[rb] = lo;
        skip_n[rb] = n;
        prefix[rb + 1] = prefix[rb] + ntile_cols - n;
    }
    const int total_tiles = prefix[nrb];
    int grid = ctx->sm_count;
    if (grid > (total_tiles + 7) / 8) grid = (total_tiles + 7) / 8;
    if (grid < 1) grid = 1;

    // ---- schedule: which CTA computes which tiles, in which order ----------------------------------------------
    // The centred matrix (Npad x ld doubles; 288 MB at 600 x 50 kb) does not fit the 126 MB L2, and every tile needs
    // a 128-row A panel and a 128-row B panel of it.  With CTAs spread over unrelated columns every panel comes from
    // DRAM for every tile (measured: 188 GB per launch at 600 x 50 kb).  So work is handed out in *rounds*: in a
    // round a group of G CTAs shares one row block and walks its valid column tiles interleaved (CTA j takes tiles
    // j, j+G, ...), all groups starting at column 0 together.  The CTAs then sit on (nearly) the same B panel at the
    // same time - it is read from DRAM once per round - and the live A panels (grid/G of them) stay L2-resident.
    // Row blocks left after the last full round are cut into contiguous column ranges that level the CTAs' tile
    // counts (water-filling), so the balance of the plain equal split is kept.
    const double tile_bytes = (double)BM * ld * sizeof(double);
    const double matrix_bytes = (double)Npad * ld * sizeof(double);
    int G = ctx->k5_group;
    if (G <= 0) {
        G = 1;
        if (matrix_bytes > 64e6)
            while (G < 8 && (double)(grid / G) * tile_bytes > 48e6) G *= 2;
    }
    const bool rounds_on = matrix_bytes > 64e6 || ctx->k5_group > 0;

    // Symmetric search (whole-matrix calls): d(i, j) = d(j, i), so each unordered pair of bin blocks {I, J} needs one
    // tile, not two - the tile's scores are filtered against the ROW bins' thresholds and against the COLUMN bins'
    // thresholds, and the column side's survivors go to per-bin incoming buffers through global atomics.  That only
    // pays once thresholds are tight (an unfiltered column side would flood the buffers), hence two passes:
    //   pass A  a symmetric subset of the block pairs ((I + J) % sym_frac == 0, and the diagonal) is computed
    //           from both sides the ordinary way, rows only; every bin leaves a threshold ~ its k-th smallest distance
    //           among 1/sym_frac of all candidates;
    //   pass B  the other pairs, once each: block I takes J = I + 1 ... I + nb/2 (cyclically), so the load is level and all
    //           CTAs slide over the same window of B panels (L2-resident) at the same time.
    // Work: (1/sym_frac + (1 - 1/sym_frac) / 2) of the plain search.
    const int sym_frac = ctx->k5_sym;
    const bool sym = sym_frac >= 2 && row_begin == 0 && row_end == N && nrb >= 24;
    // symmetric pass of the tcgen05 filter: four CTAs per row block level the CTAs' finish times (measured at 600 x 50 kb,
    // profiles/tc_group_50kb_r03ab.txt: G = 1, 2, 4, 8 -> K5 3.30, 2.97, 2.77, 2.83 ms; the plain pass of a row range is
    // as fast with two)
    if (sym && ctx->k5_group <= 0 && ctx->k5_f16 == 2 && G == 2) G = 4;
    std::vector<Piece> pieces;
    std::vector<int> listA, listB, offA, offB;
    int gridA = 0, gridB = 0;
    long long tilesA = 0, tilesB = 0;
    if (!sym) {
        schedule_pieces(prefix, nrb, grid, G, rounds_on, 0, pieces);
    } else {
        const int nb = nrb;
        pair_lists(nb, skip_lo, skip_n, sym_frac, 0, nb, listA, offA, listB, offB);
        tilesA = (long long)listA.size();
        tilesB = (long long)listB.size();
        gridA = (int)std::max(1ll, std::min<long long>(ctx->sm_count, (tilesA + 7) / 8));
        gridB = (int)std::max(1ll, std::min<long long>(ctx->sm_count, (tilesB + 7) / 8));
        // pass A: contiguous split, so a row block is cut at most once or twice and every bin's threshold comes from (nearly)
        // its whole sample.  (Rounds would chop the left-over row blocks into ~20 pieces of 2-3 tiles: thresholds loose
        // enough to flood those bins' incoming buffers - measured: ~900 rows in the exhaustive fallback, +240 ms.)  The price:
        // the CTAs are out of step and pass A's B panels come from DRAM (24 GB at 600 x 50 kb) - see DESIGN.md section 7.
        schedule_pieces(offA, nb, gridA, 1, false, 0, pieces);
        int GB = G;
        if (GB > gridB) GB = gridB;
        schedule_pieces(offB, nb, gridB, GB, rounds_on, 1, pieces);
    }
    // segments (one candidate buffer set per piece) are numbered row-block-major so that K6 finds a row's pieces side by side
    // One piece table for both passes (pass A's pieces first); cta_piece_begin holds, per pass, grid+1 absolute indices.
    const int grid0 = sym ? gridA : grid;            // CTAs of the first (or only) launch
    std::vector<int> rb_seg_first(nrb, 0), rb_seg_count(nrb, 0), cta_piece_begin, piece_tab;
    // K5t keeps one segment per column half of a piece (its two epilogue warpgroups share no row state)
    const int spp = ctx->k5_f16 == 2 ? TC_SEGS_PER_PIECE : 1;
    const int npieces = (int)pieces.size();
    const int nseg = npieces * spp;
    {
        for (const Piece& pc : pieces) rb_seg_count[pc.rb] += spp;
        int run = 0;
        for (int rb = 0; rb < nrb; ++rb) { rb_seg_first[rb] = run; run += rb_seg_count[rb]; }
        std::vector<int> next(rb_seg_first);
        for (Piece& pc : pieces) { pc.seg = next[pc.rb]; next[pc.rb] += spp; }
        std::stable_sort(pieces.begin(), pieces.end(), [](const Piece& x, const Piece& y) {
            return x.pass != y.pass ? x.pass < y.pass : x.cta < y.cta;
        });
        piece_tab.resize((size_t)std::max(npieces, 1) * 5);
        std::vector<int> per_cta0(grid0 + 1, 0), per_cta1(gridB + 1, 0);
        int n0 = 0;
        for (int i = 0; i < npieces; ++i) {
            const Piece& pc = pieces[i];
            if (pc.pass == 0) { per_cta0[pc.cta + 1]++; ++n0; } else { per_cta1[pc.cta + 1]++; }
            piece_tab[(size_t)i * 5 + 0] = pc.rb;
            piece_tab[(size_t)i * 5 + 1] = pc.q0;
            piece_tab[(size_t)i * 5 + 2] = pc.q1;
            piece_tab[(size_t)i * 5 + 3] = pc.step;
            piece_tab[(size_t)i * 5 + 4] = pc.seg;
        }
        for (int c = 0; c < grid0; ++c) per_cta0[c + 1] += per_cta0[c];
        cta_piece_begin = per_cta0;
        if (sym) {
            per_cta1[0] = n0;
            for (int c = 0; c < gridB; ++c) per_cta1[c + 1] += per_cta1[c];
            cta_piece_begin.insert(cta_piece_begin.end(), per_cta1.begin(), per_cta1.end());
        }
    }
    // the symmetric search's tile lists travel behind the piece table: [offA nrb+1][offB nrb+1][listA][listB]
    std::vector<int> sym_tab;
    if (sym) {
        sym_tab.insert(sym_tab.end(), offA.begin(), offA.end());
        sym_tab.insert(sym_tab.end(), offB.begin(), offB.end());
        sym_tab.insert(sym_tab.end(), listA.begin(), listA.end());
        sym_tab.insert(sym_tab.end(), listB.begin(), listB.end());
    }

    P.row_cs.swap(row_cs); P.row_ce.swap(row_ce); P.skip_lo.swap(skip_lo); P.skip_n.swap(skip_n);
    P.rb_seg_first.swap(rb_seg_first); P.rb_seg_count.swap(rb_seg_count); P.cta_piece_begin.swap(cta_piece_begin);
    P.piece_tab.swap(piece_tab); P.sym_tab.swap(sym_tab);
    P.nrb = nrb; P.total_tiles = total_tiles; P.grid = grid; P.sym = sym ? 1 : 0; P.sym_frac = sym_frac; P.gridA = gridA; P.gridB = gridB;
    P.grid0 = grid0; P.nseg = nseg; P.tilesA = tilesA; P.tilesB = tilesB; P.listA_size = listA.size();
    {   // fingerprint of what the device copy of the metadata must hold
        unsigned long long h = 1469598103934665603ull;
        auto mix = [&](const void* p, size_t bytes) {
            const unsigned char* c = static_cast<const unsigned char*>(p);
            for (size_t i = 0; i < bytes; ++i) { h ^= c[i]; h *= 1099511628211ull; }
        };
        mix(chrom_bins_h, (size_t)nchrom * sizeof(int));
        const int dims[8] = {N, row_begin, row_end, grid0, nrb, nseg, sym ? sym_frac : 0, gridB};
        mix(dims, sizeof(dims));
        mix(P.piece_tab.data(), P.piece_tab.size() * sizeof(int));
        mix(P.cta_piece_begin.data(), P.cta_piece_begin.size() * sizeof(int));
        P.content_hash = h;
    }
    P.key = plan_key;
    P.valid = true;
    }
    const std::vector<int>& row_cs = P.row_cs; const std::vector<int>& row_ce = P.row_ce;
    const std::vector<int>& skip_lo = P.skip_lo; const std::vector<int>& skip_n = P.skip_n;
    const std::vector<int>& rb_seg_first = P.rb_seg_first; const std::vector<int>& rb_seg_count = P.rb_seg_count;
    const std::vector<int>& cta_piece_begin = P.cta_piece_begin; const std::vector<int>& piece_tab = P.piece_tab;
    const std::vector<int>& sym_tab = P.sym_tab;
    const int nrb = P.nrb, total_tiles = P.total_tiles, grid = P.grid, gridA = P.gridA, gridB = P.gridB, grid0 = P.grid0, nseg = P.nseg;
    const bool sym = P.sym != 0;
    const int sym_frac = P.sym_frac;
    const long long tilesA = P.tilesA, tilesB = P.tilesB;
    const size_t listA_size = P.listA_size;

    // ---- workspace ----------------------------------------------------------------------------------------
    double* Xc; double* norms; int* d_row_cs; int* d_row_ce; int* d_meta;
    u64* cand_key; int* cand_j; int* seg_cnt; int* seg_flag; int* slow;
    int rc;
    // (the fp16 matrix of K5t - rows of S + 4 halves padded to whole chunks, plus one more chunk - can exceed it for tiny S)
    if ((rc = wc_reserve(ctx, SLOT_XC, std::max(Npad * ld * sizeof(double), Npad * ((size_t)(S + 4 + 2 * BKH) / BKH * BKH + BKH) * sizeof(__half)), (void**)&Xc))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_NORMS, Npad * sizeof(double), (void**)&norms))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_ROWCS, (size_t)N * sizeof(int), (void**)&d_row_cs))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_ROWCE, (size_t)N * sizeof(int), (void**)&d_row_ce))) return rc;
    const size_t meta_ints = 4 * (size_t)nrb + cta_piece_begin.size() + piece_tab.size() + sym_tab.size();
    if ((rc = wc_reserve(ctx, SLOT_RBMETA, meta_ints * sizeof(int), (void**)&d_meta))) return rc;
    const size_t cand_n = (size_t)std::max(nseg, 1) * BM * cap;
    if ((rc = wc_reserve(ctx, SLOT_CAND_D, cand_n * sizeof(u64), (void**)&cand_key))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_CAND_J, cand_n * sizeof(int), (void**)&cand_j))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_SEGCNT, (size_t)std::max(nseg, 1) * BM * sizeof(int), (void**)&seg_cnt))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_SEGFLAG, (size_t)std::max(nseg, 1) * BM * sizeof(int), (void**)&seg_flag))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_SLOW, ((size_t)rows + 1) * sizeof(int), (void**)&slow))) return rc;
    u64* row_thr;
    const size_t thr_n = (size_t)nrb * BM + BN;            // padded: the symmetric pass reads whole column tiles of it
    if ((rc = wc_reserve(ctx, SLOT_ROWTHR, thr_n * sizeof(u64), (void**)&row_thr))) return rc;
    u64* in_key = nullptr; int* in_j = nullptr; int* in_cnt = nullptr;
    // a bin's threshold after pass A lets through ~ k * sym_frac / 2 of the column-side scores; 4x head room
    int in_cap = 0;
    if (sym) {
        in_cap = 256;
        while (in_cap < 2 * k * sym_frac) in_cap *= 2;
        if ((rc = wc_reserve(ctx, SLOT_IN_KEY, (size_t)rows * in_cap * sizeof(u64), (void**)&in_key))) return rc;
        if ((rc = wc_reserve(ctx, SLOT_IN_J, (size_t)rows * in_cap * sizeof(int), (void**)&in_j))) return rc;
        if ((rc = wc_reserve(ctx, SLOT_IN_CNT, (size_t)rows * sizeof(int), (void**)&in_cnt))) return rc;
    }
    int* d_skip_lo = d_meta;
    int* d_skip_n = d_skip_lo + nrb;
    int* d_seg_first = d_skip_n + nrb;
    int* d_seg_count = d_seg_first + nrb;
    int* d_cta_piece = d_seg_count + nrb;
    int* d_pieces = d_cta_piece + cta_piece_begin.size();
    int* d_sym = d_pieces + piece_tab.size();

    {
        // repeated calls on the same problem find the metadata on the device already
        unsigned long long h = P.content_hash;
        const unsigned long long ptrs[2] = {(unsigned long long)(uintptr_t)d_row_cs, (unsigned long long)(uintptr_t)d_meta};
        for (int i = 0; i < 2; ++i) { h ^= ptrs[i]; h *= 1099511628211ull; }
        if (h != ctx->sched_hash) {
            WC_CUDA(cudaMemcpyAsync(d_row_cs, row_cs.data(), (size_t)N * sizeof(int), cudaMemcpyHostToDevice, stream));
            WC_CUDA(cudaMemcpyAsync(d_row_ce, row_ce.data(), (size_t)N * sizeof(int), cudaMemcpyHostToDevice, stream));
            WC_CUDA(cudaMemcpyAsync(d_skip_lo, skip_lo.data(), (size_t)nrb * sizeof(int), cudaMemcpyHostToDevice, stream));
            WC_CUDA(cudaMemcpyAsync(d_skip_n, skip_n.data(), (size_t)nrb * sizeof(int), cudaMemcpyHostToDevice, stream));
            WC_CUDA(cudaMemcpyAsync(d_seg_first, rb_seg_first.data(), (size_t)nrb * sizeof(int), cudaMemcpyHostToDevice, stream));
            WC_CUDA(cudaMemcpyAsync(d_seg_count, rb_seg_count.data(), (size_t)nrb * sizeof(int), cudaMemcpyHostToDevice, stream));
            WC_CUDA(cudaMemcpyAsync(d_cta_piece, cta_piece_begin.data(), cta_piece_begin.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
            WC_CUDA(cudaMemcpyAsync(d_pieces, piece_tab.data(), piece_tab.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
            if (sym)
                WC_CUDA(cudaMemcpyAsync(d_sym, sym_tab.data(), sym_tab.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
            ctx->sched_hash = h;
        }
    }
    WC_CUDA(cudaMemsetAsync(slow, 0, sizeof(int), stream));
    WC_CUDA(cudaMemsetAsync(seg_cnt, 0, (size_t)std::max(nseg, 1) * BM * sizeof(int), stream));
    WC_CUDA(cudaMemsetAsync(seg_flag, 0, (size_t)std::max(nseg, 1) * BM * sizeof(int), stream));
    if (sym) WC_CUDA(cudaMemsetAsync(in_cnt, 0, (size_t)rows * sizeof(int), stream));

    // ---- K4 -------------------------------------------------------------------------------------------------
    // Option k5_f16: the filter runs on the fp16 tensor cores (K4h + K5h); falls back to the fp64 filter when the matrix
    // holds finite values fp16 cannot represent.
    bool f16 = ctx->k5_f16 != 0;
    const bool tc = ctx->k5_f16 == 2;          // tcgen05 / TMEM filter (K5t); 1 = mma.sync filter (K5h)
    // K5t folds the norms into the contraction: four more columns, and a second version of the last chunk (wc_prepare_f16_kernel)
    const int ldh = tc ? (S + 4 + BKH - 1) / BKH * BKH : (S + BKH - 1) / BKH * BKH;
    const int ldx = tc ? ldh + BKH : ldh;                 // row stride of the fp16 matrix, in halves
    float* n32 = nullptr;
    double nmax = 0.0;
    // error of the fp16 filter: |d~ - d| <= eps * (n_i + n_j) + sub; eps = operand rounding (2 x 2^-11), fp32 accumulation
    // of ldh products (taken one bit worse than IEEE; twice that with the norms among the summands: the partial sums are
    // bounded by n_i + n_j instead of half of it), the norms' two-half split and the fp32 compare (2^-20)
    const double eps16 = ldexp(1.0, -10) * (1.0 + ldexp(1.0, -11)) + (tc ? 2.0 : 1.0) * (double)ldh * ldexp(1.0, -23) +
                         (tc ? ldexp(1.0, -20) : ldexp(1.0, -21));
    const unsigned long long* f16_stats_d = nullptr;       // set: K4h's range flag is checked at the end of the call
    WC_CUDA(cudaEventRecord(ctx->ev[0], stream));
    if (f16) {
        unsigned long long* stats;
        if ((rc = wc_reserve(ctx, SLOT_N32, Npad * sizeof(float), (void**)&n32))) return rc;
        if ((rc = wc_reserve(ctx, SLOT_F16STAT, 4 * sizeof(unsigned long long), (void**)&stats))) return rc;
        WC_CUDA(cudaMemsetAsync(stats, 0, 2 * sizeof(unsigned long long), stream));
        wc_prepare_f16_kernel<<<(int)((Npad * 32 + 255) / 256), 256, 0, stream>>>(corrected_d, N, (int)Npad, S, ldh, ldx, tc ? 1 : 0,
                                                                                  reinterpret_cast<__half*>(Xc), norms, n32, stats);
        WC_CUDA(cudaGetLastError());
        if (ctx->k5_f16_checked != 0) {
            // the range check and the largest norm come back at the end of the call (with the fallback-row counter): no
            // host round trip between K4h and K5; a matrix outside fp16's range repeats the call with the fp64 filter
            f16_stats_d = stats;
            wc_f16_margin_kernel<<<1, 1, 0, stream>>>(stats, S, eps16, reinterpret_cast<double*>(stats + 2));
        } else {
            unsigned long long st_h[2] = {0, 0};
            WC_CUDA(cudaMemcpyAsync(st_h, stats, sizeof(st_h), cudaMemcpyDeviceToHost, stream));
            WC_CUDA(cudaStreamSynchronize(stream));
            memcpy(&nmax, &st_h[0], sizeof(double));
            if (st_h[1] != 0) f16 = false;            // |x - 1| > 60000 somewhere: outside fp16's range
        }
    }
    if (!f16) {
        const int blocks = (int)((Npad * 32 + 255) / 256);
        wc_prepare_kernel<<<blocks, 256, 0, stream>>>(corrected_d, N, (int)Npad, S, ld, Sx, Xc, norms);
    }
    WC_CUDA(cudaGetLastError());
    WC_CUDA(cudaEventRecord(ctx->ev[1], stream));
    // error of the fp16 filter: |d~ - d| <= eps * (n_i + n_j) + sub; eps = operand rounding (2 x 2^-11), fp32 accumulation
    // of ldh products (taken one bit worse than IEEE), the fp32 epilogue; sub = fp16 subnormal spacing on tiny values
    const double filt_mcoef = f16 ? 2.0 * eps16 : mcoef;
    const double filt_madd = f16 ? 2.0 * eps16 * nmax + ldexp(1.0, -20) * sqrt((double)S * nmax) : 0.0;

    // ---- K5 -------------------------------------------------------------------------------------------------
    CUtensorMap tmap;
    {
        if (!ctx->encode_tiled) {
            wc_set_error("cuTensorMapEncodeTiled is not available from this driver");
            return WC_ERR_CUDA;
        }
        cuuint64_t dims[2] = {(cuuint64_t)(f16 ? ldx : ld), (cuuint64_t)Npad};
        cuuint64_t strides[1] = {f16 ? (cuuint64_t)ldx * sizeof(__half) : (cuuint64_t)ld * sizeof(double)};
        cuuint32_t box[2] = {(cuuint32_t)(f16 ? BKH : BK), BM};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = reinterpret_cast<PFN_encodeTiled>(ctx->encode_tiled)(
            &tmap, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, Xc, dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            wc_set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
            return WC_ERR_CUDA;
        }
    }
    TopkArgs ta;
    ta.norms = norms; ta.row_cs = d_row_cs; ta.row_ce = d_row_ce; ta.N = N;
    ta.row_begin = row_begin; ta.row_end = row_end; ta.nkc = nkc; ta.nd_last = nd_last; ta.extra_h = extra_h;
    ta.rb_skip_lo = d_skip_lo; ta.rb_skip_n = d_skip_n; ta.nrb = nrb;
    ta.cta_piece_begin = d_cta_piece; ta.pieces = d_pieces;
    ta.cand_key = cand_key; ta.cand_j = cand_j; ta.seg_cnt = seg_cnt; ta.seg_flag = seg_flag;
    ta.cap = cap; ta.k = k; ta.mcoef = filt_mcoef; ta.tau_init = f16 ? 3e38 : 1e10 * (1.0 + 1e-6);
    ta.row_thr = row_thr;
    ta.lag = ctx->k5_lag;
    ta.nstages = cap <= 512 ? (sym ? 4 : 5) : 3;          // the symmetric pass keeps 8 KiB of column thresholds in shared memory
    if (f16) { ta.nstages = 4; ta.nkc = ldh / BKH; }
    ta.kb_last = f16 ? (tc ? ldh : ldh - BKH) : 0;
    if (ctx->k5_stages >= 3 && ctx->k5_stages <= MAX_STAGES) ta.nstages = ctx->k5_stages;
    ta.tile_list = nullptr; ta.rb_list_off = nullptr; ta.final_prune = sym ? 1 : 0;
    ta.in_key = in_key; ta.in_j = in_j; ta.in_cnt = in_cnt; ta.in_cap = in_cap; ta.col_thr = row_thr;
    ta.madd = filt_madd; ta.n32 = n32;
    ta.madd_p = f16_stats_d != nullptr ? reinterpret_cast<const double*>(f16_stats_d + 2) : nullptr;
    ta.dbg = f16 && tc ? ctx->dbg_scores : nullptr; ta.dbg_ld = ctx->dbg_ld;
    ta.prof = nullptr;
    ta.trace = nullptr;
    const int grid_prof = sym ? std::max(gridA, gridB) : grid;
    if (ctx->debug_profile) {
        if ((rc = wc_reserve(ctx, SLOT_PROF, ((size_t)grid_prof * 8 + 512) * sizeof(long long), (void**)&ta.prof))) return rc;
        WC_CUDA(cudaMemsetAsync(ta.prof, 0, ((size_t)grid_prof * 8 + 512) * sizeof(long long), stream));
        ta.trace = ta.prof + (size_t)grid_prof * 8;
    }
    const size_t topk_smem_legacy = f16
        ? (size_t)ta.nstages * STAGE_BYTES + sizeof(TopkState) + (size_t)CONSUMER_WARPS * F16_SCRATCH +
              (size_t)CONSUMER_WARPS * (BN * sizeof(u64) + STG * sizeof(uint4) + (2 * BN + 32) * sizeof(float))
        : (size_t)ta.nstages * STAGE_BYTES + sizeof(TopkState) +
              (size_t)CONSUMER_WARPS * std::max<size_t>((size_t)cap * 12, 8192) +
              (sym ? (size_t)CONSUMER_WARPS * (BN * sizeof(u64) + STG * sizeof(uint4)) : 0);
    const bool use_tc = f16 && tc;
    const size_t topk_smem = use_tc ? TC_SMEM_BYTES : topk_smem_legacy;
    if (topk_smem > 227 * 1024) { wc_set_error("K5 shared memory %zu exceeds 227 KiB", topk_smem); return WC_ERR_INTERNAL; }
    const bool dbg = use_tc && ta.dbg != nullptr;
    {   // opt in to the large dynamic shared memory for every kernel this call may launch
        const int sm_bytes = (int)topk_smem;
        if (use_tc) {
            WC_CUDA(cudaFuncSetAttribute(wc_dist_topk_tc_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
            WC_CUDA(cudaFuncSetAttribute(wc_dist_topk_tc_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
            if (dbg) {
                WC_CUDA(cudaFuncSetAttribute(wc_dist_topk_tc_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
                WC_CUDA(cudaFuncSetAttribute(wc_dist_topk_tc_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
            }
        } else if (f16) {
            WC_CUDA(cudaFuncSetAttribute(wc_dist_topk_f16_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
            WC_CUDA(cudaFuncSetAttribute(wc_dist_topk_f16_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
        } else {
            WC_CUDA(cudaFuncSetAttribute(wc_dist_topk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
            WC_CUDA(cudaFuncSetAttribute(wc_dist_topk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
        }
    }
    wc_fill_u64_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, stream>>>(row_thr, (size_t)rows, host_key_of_tau(ta.tau_init));
    wc_fill_u64_kernel<<<(unsigned)((thr_n - rows + 255) / 256), 256, 0, stream>>>(row_thr + rows, thr_n - (size_t)rows, KEY_NEVER);
    WC_CUDA(cudaEventRecord(ctx->ev[2], stream));
    ta.coln32 = n32; ta.col_ids = nullptr;
    // K5t takes a second tensor map for the column operand (the pivot pass reads a different matrix); the legacy kernels one
    auto launch = [&](bool symmetric, int g) {
        if (use_tc) {
            auto kern = symmetric ? (dbg ? wc_dist_topk_tc_kernel<1, true> : wc_dist_topk_tc_kernel<1, false>)
                                  : (dbg ? wc_dist_topk_tc_kernel<0, true> : wc_dist_topk_tc_kernel<0, false>);
            kern<<<g, TC_THREADS, topk_smem, stream>>>(tmap, tmap, ta);
        } else if (f16) {
            if (symmetric) wc_dist_topk_f16_kernel<true><<<g, TOPK_THREADS, topk_smem, stream>>>(tmap, ta);
            else wc_dist_topk_f16_kernel<false><<<g, TOPK_THREADS, topk_smem, stream>>>(tmap, ta);
        } else {
            if (symmetric) wc_dist_topk_kernel<true><<<g, TOPK_THREADS, topk_smem, stream>>>(tmap, ta);
            else wc_dist_topk_kernel<false><<<g, TOPK_THREADS, topk_smem, stream>>>(tmap, ta);
        }
    };
    long long pivot_launches = 0;
    // pivot pass (K5t): every target bin of the call starts the search proper with a threshold close to its final one
    const int R = (use_tc && !dbg && ctx->k5_pivots != 0 && rows >= 2 * BM) ? pivot_count(N, k) : 0;
    if (R > 0) {
        if ((rc = tc_pivot_pass(ctx, stream, tmap, ta, reinterpret_cast<const __half*>(Xc), ldh, ldx, N, nrb, rb_seg_first, R))) return rc;
        pivot_launches = 3;
    }
    WC_CUDA(cudaEventRecord(ctx->ev[17], stream));
    if (!sym) {
        launch(false, grid);
    } else {
        const int nb1 = nrb + 1;
        ta.tile_list = d_sym + 2 * nb1;                                  // pass A
        ta.rb_list_off = d_sym;
        launch(false, gridA);
        WC_CUDA(cudaGetLastError());
        WC_CUDA(cudaEventRecord(ctx->ev[16], stream));
        ta.tile_list = d_sym + 2 * nb1 + (int)listA_size;              // pass B
        ta.rb_list_off = d_sym + nb1;
        ta.cta_piece_begin = d_cta_piece + (gridA + 1);
        launch(true, gridB);
    }
    WC_CUDA(cudaGetLastError());
    WC_CUDA(cudaEventRecord(ctx->ev[3], stream));

    // ---- K6 -------------------------------------------------------------------------------------------------
    FinArgs fa;
    fa.X = corrected_d; fa.N = N; fa.S = S; fa.norms = norms; fa.row_cs = d_row_cs; fa.row_ce = d_row_ce;
    fa.row_begin = row_begin; fa.row_end = row_end; fa.rb_seg_first = d_seg_first; fa.rb_seg_count = d_seg_count;
    fa.cand_key = cand_key; fa.cand_j = cand_j; fa.seg_cnt = seg_cnt; fa.seg_flag = seg_flag; fa.cap = cap; fa.k = k;
    fa.shortcap = k <= (f16 ? 96 : 128) ? 256 : 512;          // the fp16 filter's wider window lets ~10-25 % more through
    fa.mcoef = filt_mcoef; fa.idx_out = idx_d; fa.dist_out = dist_d; fa.slow_list = slow + 1; fa.slow_count = slow;
    fa.vec = (S % 4 == 0 && (reinterpret_cast<uintptr_t>(corrected_d) & 31) == 0) ? 4 : 1;
    fa.in_key = in_key; fa.in_j = in_j; fa.in_cnt = in_cnt; fa.in_cap = in_cap; fa.in_nsrc = 1; fa.in_src_rows = 0;
    fa.madd = filt_madd; fa.row_thr = row_thr; fa.madd_p = ta.madd_p;
    fa.slow_bias = 0;
    WC_CUDA(cudaEventRecord(ctx->ev[4], stream));
    long long fin_launches = 0;
    // Called from wc_newref_topk_host: K6 runs in k6_parts row ranges and every finished range but the last travels to the
    // host (a non-blocking stream behind an event) while the next one is re-scored - the copy left at the end is
    // 1 / k6_parts of the table.
    const int nparts = (ctx->d2h_idx_h != nullptr && rows >= 16 * BM) ? std::max(1, ctx->k6_parts) : 1;
    ctx->d2h_rows_done = 0;
    for (int pi = 0, r0 = 0; pi < nparts; ++pi) {
        const int r1 = pi + 1 == nparts ? (int)rows : (int)((long long)rows * (pi + 1) / nparts) / BM * BM;
        if (r1 <= r0) continue;
        FinArgs f = fa;
        const int hb = r0 / BM;
        f.row_begin = row_begin + r0; f.row_end = row_begin + r1;
        f.rb_seg_first += hb; f.rb_seg_count += hb;
        f.idx_out += (size_t)r0 * k; f.dist_out += (size_t)r0 * k;
        f.slow_bias = r0;
        if (f.row_thr != nullptr) f.row_thr += r0;
        if (f.in_key != nullptr) { f.in_key += (size_t)r0 * in_cap; f.in_j += (size_t)r0 * in_cap; f.in_cnt += r0; }
        long long l = 0;
        if ((rc = launch_finalize(ctx, stream, f, r1 - r0, f16 != 0, &l))) return rc;
        fin_launches += l;
        if (pi + 1 < nparts) {
            WC_CUDA(cudaEventRecord(ctx->d2h_ev, stream));
            WC_CUDA(cudaStreamWaitEvent(ctx->d2h_stream, ctx->d2h_ev, 0));
            WC_CUDA(cudaMemcpyAsync(ctx->d2h_idx_h + (size_t)r0 * k, idx_d + (size_t)r0 * k, (size_t)(r1 - r0) * k * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->d2h_stream));
            WC_CUDA(cudaMemcpyAsync(ctx->d2h_dist_h + (size_t)r0 * k, dist_d + (size_t)r0 * k, (size_t)(r1 - r0) * k * sizeof(double), cudaMemcpyDeviceToHost, ctx->d2h_stream));
            ctx->d2h_rows_done = (size_t)r1;
        }
        r0 = r1;
    }
    WC_CUDA(cudaEventRecord(ctx->ev[5], stream));

    int nslow = 0, k6_stats[4] = {0, 0, 0, 0};
    WC_CUDA(cudaMemcpyAsync(&nslow, slow, sizeof(int), cudaMemcpyDeviceToHost, stream));
    if (ctx->k6_stats_d != nullptr) WC_CUDA(cudaMemcpyAsync(k6_stats, ctx->k6_stats_d, 4 * sizeof(int), cudaMemcpyDeviceToHost, stream));
    unsigned long long f16_flag = 0;
    if (f16_stats_d != nullptr) WC_CUDA(cudaMemcpyAsync(&f16_flag, f16_stats_d + 1, sizeof(f16_flag), cudaMemcpyDeviceToHost, stream));
    WC_CUDA(cudaStreamSynchronize(stream));
    if (f16_flag != 0) {                                 // |x - 1| > 60000 somewhere: outside fp16's range - the fp64 filter
        const int keep = ctx->k5_f16;
        ctx->k5_f16 = 0;
        rc = wc_newref_topk(ctx, corrected_d, N, S, chrom_bins_h, nchrom, row_begin, row_end, refsize, idx_d, dist_d, stream_v);
        ctx->k5_f16 = keep;
        return rc;
    }
    ctx->counter[8] = k6_stats[1];                       // K6 split form: live entries / shortlisted candidates over all rows
    ctx->counter[9] = k6_stats[2];
    ctx->counter[10] = k6_stats[0];
    ctx->counter[11] = k6_stats[3];
    long long launches = (sym ? 5 : 4) + pivot_launches + fin_launches;   // two fills, K4, K5 (one or two passes; pivot select + gather + pass), K6 (1 fused, or reset + select + re-score + rank)
    if (nslow > 0) {
        ctx->d2h_rows_done = 0;                          // rows of the first half may be among them: the host copies everything again
        const int batch = 64;
        double* scratch;
        if ((rc = wc_reserve(ctx, SLOT_SCRATCH, (size_t)std::min(nslow, batch) * N * sizeof(double), (void**)&scratch)))
            return rc;
        WC_CUDA(cudaEventRecord(ctx->ev[6], stream));
        for (int off = 0; off < nslow; off += batch) {
            ExhArgs ea;
            ea.X = corrected_d; ea.N = N; ea.S = S; ea.row_cs = d_row_cs; ea.row_ce = d_row_ce; ea.row_begin = row_begin;
            ea.slow_list = slow + 1; ea.list_off = off; ea.scratch = scratch; ea.k = k; ea.idx_out = idx_d; ea.dist_out = dist_d;
            wc_exhaustive_kernel<<<std::min(batch, nslow - off), EXH_THREADS, 0, stream>>>(ea);
            ++launches;
        }
        WC_CUDA(cudaGetLastError());
        WC_CUDA(cudaEventRecord(ctx->ev[7], stream));
        WC_CUDA(cudaStreamSynchronize(stream));
    }
    float ms;
    WC_CUDA(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1])); ctx->phase_ms[0] = ms;
    WC_CUDA(cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3])); ctx->phase_ms[1] = ms;
    ctx->phase_ms[8] = 0.0;
    if (sym) { WC_CUDA(cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[16])); ctx->phase_ms[8] = ms; }
    WC_CUDA(cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5])); ctx->phase_ms[2] = ms;
    if (nslow > 0) { WC_CUDA(cudaEventElapsedTime(&ms, ctx->ev[6], ctx->ev[7])); ctx->phase_ms[3] = ms; }
    ctx->counter[0] = launches;
    ctx->counter[1] = nslow;
    ctx->counter[2] = total_tiles;                       // tiles the plain search computes (= counter 3 unless symmetric)
    ctx->counter[3] = sym ? tilesA + tilesB : total_tiles;
    ctx->counter[4] = sym ? std::max(gridA, gridB) : grid;
    ctx->counter[7] = (f16 ? ctx->k5_f16 : 0) | (R << 4);
    return WC_OK;
}

extern "C" int wc_newref_topk_host(wc_ctx* ctx, const double* corrected_h, int N, int S, const int* chrom_bins_h,
                                   int nchrom, int row_begin, int row_end, int refsize, int32_t* idx_h,
                                   double* dist_h) {
    WC_CHECK_ARG(ctx != nullptr && corrected_h != nullptr);
    WC_CHECK_ARG(N > 0 && S > 0 && refsize >= 1);
    WC_CHECK_ARG(row_begin >= 0 && row_begin <= row_end && row_end <= N);
    WC_CUDA(cudaSetDevice(ctx->device));
    const size_t rows = (size_t)(row_end - row_begin);
    double* X; int32_t* idx; double* dist;
    int rc;
    if ((rc = wc_reserve(ctx, SLOT_IO_X, (size_t)N * S * sizeof(double), (void**)&X))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_IO_IDX, std::max<size_t>(rows, 1) * refsize * sizeof(int32_t), (void**)&idx))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_IO_DIST, std::max<size_t>(rows, 1) * refsize * sizeof(double), (void**)&dist))) return rc;
    WC_CUDA(cudaMemcpyAsync(X, corrected_h, (size_t)N * S * sizeof(double), cudaMemcpyHostToDevice, 0));
    if (rows) WC_CHECK_ARG(idx_h != nullptr && dist_h != nullptr);
    if (ctx->d2h_stream == nullptr) {
        WC_CUDA(cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
        WC_CUDA(cudaEventCreateWithFlags(&ctx->d2h_ev, cudaEventDisableTiming));
    }
    ctx->d2h_idx_h = idx_h; ctx->d2h_dist_h = dist_h; ctx->d2h_rows_done = 0;       // lets the search start the copy of its first half early
    rc = wc_newref_topk(ctx, X, N, S, chrom_bins_h, nchrom, row_begin, row_end, refsize, idx, dist, nullptr);
    const size_t done = rc ? 0 : ctx->d2h_rows_done;
    ctx->d2h_idx_h = nullptr; ctx->d2h_dist_h = nullptr; ctx->d2h_rows_done = 0;
    if (rc) { cudaStreamSynchronize(ctx->d2h_stream); return rc; }
    if (done == 0) WC_CUDA(cudaStreamSynchronize(ctx->d2h_stream));      // an early copy that was called off must not land after the final one
    if (rows) {
        WC_CUDA(cudaMemcpyAsync(idx_h + done * refsize, idx + done * refsize, (rows - done) * refsize * sizeof(int32_t), cudaMemcpyDeviceToHost, 0));
        WC_CUDA(cudaMemcpyAsync(dist_h + done * refsize, dist + done * refsize, (rows - done) * refsize * sizeof(double), cudaMemcpyDeviceToHost, 0));
        WC_CUDA(cudaStreamSynchronize(0));
        WC_CUDA(cudaStreamSynchronize(ctx->d2h_stream));
    }
    return WC_OK;
}

extern "C" int wc_newref_topk_wide(wc_ctx* ctx, const double* corrected_d, int N, int S, const int* chrom_bins_h,
                                   int nchrom, int row_begin, int row_end, int refsize, int32_t* idx_d, double* dist_d,
                                   void* stream_v) {
    WC_CHECK_ARG(ctx != nullptr);
    WC_CHECK_ARG(corrected_d != nullptr && chrom_bins_h != nullptr);
    WC_CHECK_ARG(N > 0 && S > 0 && nchrom > 0);
    WC_CHECK_ARG(refsize >= 1 && refsize <= WC_WIDE_REFSIZE_MAX);
    WC_CHECK_ARG(row_begin >= 0 && row_begin <= row_end && row_end <= N);
    long long tot = 0;
    for (int c = 0; c < nchrom; ++c) {
        WC_CHECK_ARG(chrom_bins_h[c] >= 0);
        tot += chrom_bins_h[c];
    }
    WC_CHECK_ARG(tot == N);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    WC_CUDA(cudaSetDevice(ctx->device));
    for (int i = 0; i < 4; ++i) ctx->phase_ms[i] = 0.0;
    for (int i = 0; i < 5; ++i) ctx->counter[i] = 0;
    ctx->timed_mask &= ~0xfu;
    const int rows = row_end - row_begin;
    if (rows == 0) return WC_OK;
    WC_CHECK_ARG(idx_d != nullptr && dist_d != nullptr);

    // exclusion range [cs, ce) of every bin: its own chromosome
    std::vector<int> rc_h(2 * (size_t)N);
    for (int c = 0, pos = 0; c < nchrom; pos += chrom_bins_h[c++])
        for (int i = 0; i < chrom_bins_h[c]; ++i) { rc_h[pos + i] = pos; rc_h[(size_t)N + pos + i] = pos + chrom_bins_h[c]; }
    // rows per chunk: a multiple of 128 whose distances fit WIDE_CHUNK_BYTES (at least 128)
    const size_t row_bytes = (size_t)N * sizeof(double);
    int R = (int)std::min<size_t>(WIDE_CHUNK_BYTES / row_bytes / 128 * 128, (size_t)(rows + 127) / 128 * 128);
    if (R < 128) R = 128;
    int* rc_d;
    double* D;
    int rc;
    if ((rc = wc_reserve(ctx, SLOT_WIDE_ROWS, rc_h.size() * sizeof(int), (void**)&rc_d))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_WIDE_D, (size_t)R * row_bytes, (void**)&D))) return rc;
    WC_CUDA(cudaMemcpyAsync(rc_d, rc_h.data(), rc_h.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
    int P = 32;
    while (P < refsize) P <<= 1;
    const size_t smem = (size_t)P * (sizeof(u64) + sizeof(int));
    WC_CUDA(cudaFuncSetAttribute(wc_wide_rank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));

    WideRankArgs ra;
    ra.D = D;
    ra.N = N;
    ra.k = refsize;
    ra.row_cs = rc_d;
    ra.row_ce = rc_d + N;
    double ms_dist = 0.0, ms_rank = 0.0;
    long long launches = 0;
    for (int c0 = row_begin; c0 < row_end; c0 += R) {
        const int r = std::min(R, row_end - c0);
        WC_CUDA(cudaEventRecord(ctx->ev[0], stream));
        const dim3 grid((N + WIDE_TILE - 1) / WIDE_TILE, (r + WIDE_TILE - 1) / WIDE_TILE);
        wc_wide_dist_kernel<<<grid, WIDE_DIST_THREADS, 0, stream>>>(corrected_d, N, S, c0, r, rc_d, rc_d + N, D);
        WC_CUDA(cudaGetLastError());
        WC_CUDA(cudaEventRecord(ctx->ev[1], stream));
        ra.row0 = c0;
        ra.idx_out = idx_d + (size_t)(c0 - row_begin) * refsize;
        ra.dist_out = dist_d + (size_t)(c0 - row_begin) * refsize;
        wc_wide_rank_kernel<<<r, WIDE_RANK_THREADS, smem, stream>>>(ra);
        WC_CUDA(cudaGetLastError());
        WC_CUDA(cudaEventRecord(ctx->ev[2], stream));
        WC_CUDA(cudaEventSynchronize(ctx->ev[2]));        // per-chunk phase times (the call is synchronous anyway)
        float ms = 0.f;
        WC_CUDA(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1])); ms_dist += ms;
        WC_CUDA(cudaEventElapsedTime(&ms, ctx->ev[1], ctx->ev[2])); ms_rank += ms;
        launches += 2;
    }
    ctx->phase_ms[1] = ms_dist;
    ctx->phase_ms[2] = ms_rank;
    ctx->counter[0] = launches;
    ctx->counter[2] = R;
    return WC_OK;
}

#include "wc_search_shard.cuh"    // sharded symmetric search (wc_newref_shard_*)

// Debug: enable per-CTA cycle counters in K5 and read them back (grid x 8 int64: total, wait-on-TMA, epilogue,
// prune, tiles, prunes, emitted entries of consumer thread 0, reserved).  Returns the number of CTAs copied.
extern "C" int wc_debug_profile(wc_ctx* ctx, int enable, long long* out_h, int max_ctas) {
    WC_CHECK_ARG(ctx != nullptr);
    ctx->debug_profile = enable;
    if (out_h == nullptr || max_ctas <= 0) return 0;
    int grid = (int)ctx->counter[4];
    if (grid > max_ctas) grid = max_ctas;
    if (grid <= 0 || ctx->buf[SLOT_PROF].p == nullptr) return 0;
    WC_CUDA(cudaMemcpy(out_h, ctx->buf[SLOT_PROF].p, (size_t)grid * 8 * sizeof(long long), cudaMemcpyDeviceToHost));
    if (max_ctas >= grid + 64)   // room for the CTA-0 timeline: 512 more int64 right after the per-CTA counters
        WC_CUDA(cudaMemcpy(out_h + (size_t)grid * 8, (long long*)ctx->buf[SLOT_PROF].p + (size_t)ctx->counter[4] * 8,
                           512 * sizeof(long long), cudaMemcpyDeviceToHost));
    return grid;
}

// Debug: the next searches with the tcgen05 filter (k5_f16 = 2) also store every filter distance d~(i, j) they compute into
// out_d[(i - row_begin) * ld + j] (float, device memory owned by the caller; j < ld).  NULL switches it off.
extern "C" int wc_debug_filter_scores(wc_ctx* ctx, float* out_d, int ld) {
    WC_CHECK_ARG(ctx != nullptr && (out_d == nullptr || ld > 0));
    ctx->dbg_scores = out_d;
    ctx->dbg_ld = out_d ? ld : 0;
    return WC_OK;
}

// Debug: the pivot selection of K5t alone - the R bins of smallest norm (ties by bin), sorted by bin (device pointers).
extern "C" int wc_debug_pivot_select(wc_ctx* ctx, const float* n32_d, int N, int R, int* ids_d) {
    WC_CHECK_ARG(ctx != nullptr && n32_d != nullptr && ids_d != nullptr && N > 0 && R > 0 && R <= N);
    WC_CUDA(cudaSetDevice(ctx->device));
    wc_pivot_select_kernel<<<1, 1024>>>(n32_d, N, R, ids_d);
    WC_CUDA(cudaGetLastError());
    WC_CUDA(cudaDeviceSynchronize());
    return WC_OK;
}

// Tuning knobs (debug / experiments).  key "k5_lag": chunks by which the trailing consumer warps lag (0..4).
extern "C" int wc_set_option(wc_ctx* ctx, const char* key, double value) {
    WC_CHECK_ARG(ctx != nullptr && key != nullptr);
    if (strcmp(key, "k5_lag") == 0) {
        WC_CHECK_ARG(value >= 0 && value <= MAX_STAGES - 2);
        ctx->k5_lag = (int)value;
        return WC_OK;
    }
    if (strcmp(key, "k5_group") == 0) {      // CTAs sharing a row block per round (0 = automatic; 1, 2, 4, 8)
        WC_CHECK_ARG(value >= 0 && value <= 64);
        ctx->k5_group = (int)value;
        return WC_OK;
    }
    if (strcmp(key, "k5_sym") == 0) {        // symmetric search for whole-matrix calls: 0 = off, f in 2..64 = on (first pass 1/f)
        if (value != 0 && (value < 2 || value > 64)) { wc_set_error("k5_sym must be 0 or 2..64"); return WC_ERR_ARG; }
        ctx->k5_sym = (int)value;
        return WC_OK;
    }
    if (strcmp(key, "k5_f16") == 0) {        // 0: fp64 filter (DMMA); 1: fp16 filter on mma.sync (K5h); 2: fp16 filter on tcgen05 / TMEM (K5t)
        WC_CHECK_ARG(value == 0 || value == 1 || value == 2);
        ctx->k5_f16 = (int)value;
        return WC_OK;
    }
    if (strcmp(key, "k5_pivots") == 0) {     // K5t: pivot pass before a symmetric search (1 = on, 0 = off)
        ctx->k5_pivots = value != 0 ? 1 : 0;
        return WC_OK;
    }
    if (strcmp(key, "k6_split") == 0) { ctx->k6_split = value != 0 ? 1 : 0; return WC_OK; }      // K6: split (streaming re-score) / fused
    if (strcmp(key, "k6_g4") == 0) { ctx->k6_g4 = value != 0 ? 1 : 0; return WC_OK; }
    if (strcmp(key, "k6_select") == 0) { ctx->k6_select = value != 0 ? 1 : 0; return WC_OK; }
    if (strcmp(key, "k6_parts") == 0) { WC_CHECK_ARG(value >= 1 && value <= 16); ctx->k6_parts = (int)value; return WC_OK; }
    if (strcmp(key, "k6_chunk") == 0) { WC_CHECK_ARG(value >= 0 && value <= 480); ctx->k6_chunk = (int)value; return WC_OK; }
    if (strcmp(key, "k6_warps") == 0) { WC_CHECK_ARG(value >= 0 && value <= 16); ctx->k6_warps = (int)value; return WC_OK; }
    if (strcmp(key, "k6_prod") == 0) { WC_CHECK_ARG(value >= 0 && value <= 8); ctx->k6_prod = (int)value; return WC_OK; }
    if (strcmp(key, "k5_stages") == 0) {
        WC_CHECK_ARG(value == 0 || (value >= 3 && value <= MAX_STAGES));
        ctx->k5_stages = (int)value;
        return WC_OK;
    }
    wc_set_error("unknown option %s", key);
    return WC_ERR_ARG;
}
