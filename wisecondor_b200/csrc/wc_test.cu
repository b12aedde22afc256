// wisecondor_b200 - batched `test` front half on B200 (sm_100a): sample preparation and within-sample z-scores.
//
// Replaces, for a batch of B samples at once,
//   toNumpyRefFormat + applyPCA   (/root/reference/wisetools.py:267-278, 104-113)            -> K7 wc_test_prep
//   trySample / repeatTest         (/root/reference/wisetools.py:407-448)                     -> K8 wc_zscore_batch
// and, once per reference, the `index[distances[i] < cutoff]` selection and the other-chromosome concatenation
// trySample rebuilds for every chromosome (wisetools.py:420-424)                               -> wc_test_table.
//
// Data layout in HBM: the corrected test values live as T[bin][sample] ("sample-minor", leading dimension ldb = B
// rounded up to 32): a warp owns 32 consecutive samples of one target bin, so every gather of a reference bin is
// one 256-byte coalesced read shared by the warp, and the whole working set of a sample tile (N x 256 B) stays in
// the 126 MB L2 across the k gathers per bin.  Marked (aberrant) bins are -1 in a working copy, exactly as in the
// reference (wisetools.py:446).  Arithmetic follows numpy's operation order (wc_numpy_order.cuh), so z, r and the
// per-sample average sigma are bit-identical to the reference's.
#include "wc_common.cuh"
#include "wc_numpy_order.cuh"

namespace {

constexpr int ZS_WARPS = 4;             // max warps per CTA of the z-score kernel (each warp: 32 samples x 1 bin at a time)
constexpr int ZS_BINS_PER_CTA = 64;

// ---------------------------------------------------------------------------------------------------------
// gather table: table[i][0..count[i]) = global masked-bin ids of bin i's usable reference bins, in stored order
// ---------------------------------------------------------------------------------------------------------
__global__ void wc_table_kernel(const int* __restrict__ indexes, const double* __restrict__ distances, int N, int k,
                                int ldk, const int* __restrict__ row_cs, const int* __restrict__ row_ce, double cutoff,
                                int* __restrict__ table, int* __restrict__ count) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= N) return;
    const int cs = row_cs[warp], ce = row_ce[warp];
    const int nother = N - (ce - cs);
    int w = 0;
    for (int base = 0; base < k; base += 32) {
        const int m = base + lane;
        bool keep = false;
        int g = 0;
        if (m < k) {
            keep = distances[(size_t)warp * k + m] < cutoff;          // wisetools.py:424 (NaN never passes)
            int j = indexes[(size_t)warp * k + m];
            if (j < 0) j += nother;                                    // numpy's negative index wraps (filler -1)
            g = j >= cs ? j + (ce - cs) : j;                           // position in chromData -> global bin
            if (j < 0 || j >= nother) keep = false;                    // numpy would raise IndexError; never stored
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (keep) table[(size_t)warp * ldk + w + __popc(bal & ((1u << lane) - 1u))] = g;
        w += __popc(bal);
    }
    for (int m = w + lane; m < ldk; m += 32) table[(size_t)warp * ldk + m] = 0;     // defined padding
    if (lane == 0) count[warp] = w;
}

// reverse table: for every bin j the bins i that list j among their usable reference bins (CSR).  When j is marked
// in a sample, exactly these bins' statistics change in the next pass.
__global__ void wc_rev_count_kernel(const int* __restrict__ table, const int* __restrict__ count, int N, int ldk,
                                    int* __restrict__ rev_cnt) {
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (i >= N) return;
    const int c = count[i];
    for (int m = lane; m < c; m += 32) atomicAdd(&rev_cnt[table[(size_t)i * ldk + m]], 1);
}
__global__ void wc_rev_scan_kernel(const int* __restrict__ rev_cnt, int N, int* __restrict__ rev_off, int* __restrict__ cursor) {
    __shared__ int s_part[1024];
    const int tid = threadIdx.x, per = (N + 1023) / 1024;
    const int i0 = min(N, tid * per), i1 = min(N, i0 + per);
    int loc = 0;
    for (int i = i0; i < i1; ++i) loc += rev_cnt[i];
    s_part[tid] = loc;
    __syncthreads();
    if (tid == 0) {
        int run = 0;
        for (int t = 0; t < 1024; ++t) { const int v = s_part[t]; s_part[t] = run; run += v; }
        rev_off[N] = run;
    }
    __syncthreads();
    int run = s_part[tid];
    for (int i = i0; i < i1; ++i) { rev_off[i] = run; cursor[i] = run; run += rev_cnt[i]; }
}
__global__ void wc_rev_fill_kernel(const int* __restrict__ table, const int* __restrict__ count, int N, int ldk,
                                   int* __restrict__ cursor, int* __restrict__ rev_idx) {
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (i >= N) return;
    const int c = count[i];
    for (int m = lane; m < c; m += 32) rev_idx[atomicAdd(&cursor[table[(size_t)i * ldk + m]], 1)] = i;
}

// ---------------------------------------------------------------------------------------------------------
// K7: sample preparation
// ---------------------------------------------------------------------------------------------------------
__global__ void wc_totals_kernel(const int* __restrict__ counts, int Nraw, double* __restrict__ totals) {
    __shared__ long long red[8];
    const int b = blockIdx.x;
    long long acc = 0;
    for (int i = threadIdx.x; i < Nraw; i += blockDim.x) acc += counts[(size_t)b * Nraw + i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long t = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
        totals[b] = (double)t;              // integer-valued: the order of the reference's float sum is irrelevant
    }
}

// Value of masked bin n of sample b: counts are divided by the sample total (wisetools.py:275); float input is taken
// as already normalised (the applyPCA-only entry point).
template <class TIn>
__device__ __forceinline__ double prep_value(const TIn* in, int ld_in, const int* map, const double* totals, int b, int n) {
    const TIn raw = in[(size_t)b * ld_in + (map ? map[n] : n)];
    return totals ? (double)raw / totals[b] : (double)raw;
}

// proj[b][j] = sum_n (x_n - mean_n) * C[j][n]        (pca.transform, wisetools.py:109)
template <class TIn>
__global__ void wc_project_kernel(const TIn* __restrict__ in, int ld_in, const int* __restrict__ map, int N,
                                  const double* __restrict__ totals, const double* __restrict__ mean,
                                  const double* __restrict__ comps, int ncomp, double* __restrict__ proj) {
    __shared__ double red[8];
    const int b = blockIdx.x;
    for (int j = 0; j < ncomp; ++j) {
        double acc = 0.0;
        for (int n = threadIdx.x; n < N; n += blockDim.x)
            acc = fma(prep_value(in, ld_in, map, totals, b, n) - mean[n], comps[(size_t)j * N + n], acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
            proj[(size_t)b * ncomp + j] = t;
        }
        __syncthreads();
    }
}

// T[n][b] = x / (proj . C[:, n] + mean_n)              (wisetools.py:111-113), transposed to sample-minor
template <class TIn>
__global__ void wc_residual_kernel(const TIn* __restrict__ in, int ld_in, const int* __restrict__ map, int N, int B,
                                   int ldb, const double* __restrict__ totals, const double* __restrict__ mean,
                                   const double* __restrict__ comps, int ncomp, const double* __restrict__ proj,
                                   double* __restrict__ T) {
    __shared__ double tile[32][33];
    const int n0 = blockIdx.x * 32, b0 = blockIdx.y * 32;
    {
        const int n = n0 + threadIdx.x, b = b0 + threadIdx.y;
        double v = 1.0;                      // padding samples: harmless finite values
        if (n < N && b < B) {
            const double x = prep_value(in, ld_in, map, totals, b, n);
            if (ncomp > 0) {
                double recon = 0.0;
                for (int j = 0; j < ncomp; ++j) recon = fma(proj[(size_t)b * ncomp + j], comps[(size_t)j * N + n], recon);
                v = x / (recon + mean[n]);
            } else {
                v = x;
            }
        }
        tile[threadIdx.x][threadIdx.y] = v;
    }
    __syncthreads();
    const int n = n0 + threadIdx.y, b = b0 + threadIdx.x;
    if (n < N && b < ldb) T[(size_t)n * ldb + b] = tile[threadIdx.y][threadIdx.x];
}

// ---------------------------------------------------------------------------------------------------------
// K8: one z-score pass over all (bin, sample) pairs
// ---------------------------------------------------------------------------------------------------------
struct ZArgs {
    const double* test;      // [N][ldb] numerators (never change)
    const double* copy;      // [N][ldb] working copy: marked bins hold -1
    const int* table;        // [N][k]
    const int* count;        // [N]
    int N, B, ldb, k;        // k = row stride of the table (wc_table_stride(refsize))
    double* z;               // [N][ldb]
    double* r;
    int* refsz;
    double* sd;
    const int* npairs;       // later passes: size of the dirty-pair list; the full kernel runs iff it exceeds pair_limit
    int pair_limit;
};

__device__ __forceinline__ void zs_cp_async_8(double* smem_dst, const double* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}

// ---- K8 building blocks ----------------------------------------------------------------------------------------
// Fast path (no marked / non-finite reference value for this lane): the lane streams its reference values straight from
// L2 into eight register accumulators - numpy's leaf order needs no storage when nothing is dropped - once for the mean
// and once more for sum((x - mean)^2).  DEV selects the second form.  `worst` collects the largest high word seen
// (sign set or exponent all ones <=> the value is not a finite number >= +0).  n <= 128.
template <bool DEV>
__device__ __forceinline__ double zs_stream_leaf(const double* cp, const int* tab, int n, size_t ldb, double mean,
                                                 unsigned& worst) {
    auto term = [&](double v) {
        if (!DEV) { worst = max(worst, (unsigned)__double2hiint(v)); return v; }
        const double d = __dsub_rn(v, mean);
        return __dmul_rn(d, d);
    };
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = __dadd_rn(res, term(cp[(size_t)tab[i] * ldb]));
        return res;
    }
    double r[8];
    {
        const int4 i0 = *reinterpret_cast<const int4*>(tab), i1 = *reinterpret_cast<const int4*>(tab + 4);
        r[0] = term(cp[(size_t)i0.x * ldb]); r[1] = term(cp[(size_t)i0.y * ldb]);
        r[2] = term(cp[(size_t)i0.z * ldb]); r[3] = term(cp[(size_t)i0.w * ldb]);
        r[4] = term(cp[(size_t)i1.x * ldb]); r[5] = term(cp[(size_t)i1.y * ldb]);
        r[6] = term(cp[(size_t)i1.z * ldb]); r[7] = term(cp[(size_t)i1.w * ldb]);
    }
    const int full = n - (n & 7);
    int i = 8;
    for (; i < full; i += 8) {
        const int4 i0 = *reinterpret_cast<const int4*>(tab + i), i1 = *reinterpret_cast<const int4*>(tab + i + 4);
        double v[8];
        v[0] = cp[(size_t)i0.x * ldb]; v[1] = cp[(size_t)i0.y * ldb]; v[2] = cp[(size_t)i0.z * ldb]; v[3] = cp[(size_t)i0.w * ldb];
        v[4] = cp[(size_t)i1.x * ldb]; v[5] = cp[(size_t)i1.y * ldb]; v[6] = cp[(size_t)i1.z * ldb]; v[7] = cp[(size_t)i1.w * ldb];
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], term(v[j]));
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, term(cp[(size_t)tab[i] * ldb]));
    return res;
}
// any n <= 512 (the table stride's limit): numpy's halving above 128 elements.  A half is len/2 rounded DOWN to a multiple of
// 8 and the other half takes the rest, so a "quarter" of n = 489..512 can still exceed 128 (489 -> 240 + 249 -> 120 + 129):
// three levels are needed before every piece is a leaf.
template <bool DEV, int LEVELS>
__device__ __forceinline__ double zs_stream_split(const double* cp, const int* tab, int n, size_t ldb, double mean,
                                                  unsigned& worst) {
    if (LEVELS == 0 || n <= 128) return zs_stream_leaf<DEV>(cp, tab, n, ldb, mean, worst);
    int h = n / 2;
    h -= h & 7;
    const double a0 = zs_stream_split<DEV, (LEVELS > 0 ? LEVELS - 1 : 0)>(cp, tab, h, ldb, mean, worst);
    return __dadd_rn(a0, zs_stream_split<DEV, (LEVELS > 0 ? LEVELS - 1 : 0)>(cp, tab + h, n - h, ldb, mean, worst));
}
template <bool DEV>
__device__ __forceinline__ double zs_stream_sum(const double* cp, const int* tab, int n, size_t ldb, double mean,
                                                unsigned& worst) {
    return zs_stream_split<DEV, 3>(cp, tab, n, ldb, mean, worst);      // 3 levels: every piece of n <= 1024 is <= 128 + 7
}

// Slow path, warp-cooperative, for one lane whose reference values contain marked (-1) / negative / non-finite entries:
// all 32 lanes fetch that sample's values, the kept ones (refData[refData >= 0], wisetools.py:425) are compacted in
// order into the warp's small shared buffer, and lanes 0..7 act as numpy's eight accumulators.
__device__ __forceinline__ double zs_coop_sum(const double* buf, int n, double mean, bool dev, int lane) {
    auto term = [&](int i) {
        const double v = buf[i];
        if (!dev) return v;
        const double d = __dsub_rn(v, mean);
        return __dmul_rn(d, d);
    };
    double res = 0.0;
    if (n <= 128) {
        if (n < 8) {
            for (int i = 0; i < n; ++i) res = __dadd_rn(res, term(i));
        } else {
            const int full = n - (n & 7);
            double r = 0.0;
            if (lane < 8) {
                r = term(lane);
                for (int i = 8 + lane; i < full; i += 8) r = __dadd_rn(r, term(i));
            }
            r = __dadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 1));
            r = __dadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 2));
            r = __dadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 4));
            res = __shfl_sync(0xffffffffu, r, 0);
            for (int i = full; i < n; ++i) res = __dadd_rn(res, term(i));
        }
    } else {
        res = np_sum_thread(term, n);          // refsize > 128: every lane redundantly, numpy's recursion
    }
    return res;
}

struct ZsSlow { double mean, sd; int n; };
__device__ __forceinline__ ZsSlow zs_slow_lane(const double* copy_col, const int* tab, int cnt, size_t ldb, double* buf,
                                               int lane) {
    int n = 0;
    __syncwarp();
    for (int base = 0; base < cnt; base += 32) {
        const int m = base + lane;
        const double v = m < cnt ? copy_col[(size_t)tab[m] * ldb] : -1.0;
        const bool keep = m < cnt && v >= 0.0;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (keep) buf[n + __popc(bal & ((1u << lane) - 1u))] = v;
        n += __popc(bal);
    }
    __syncwarp();
    ZsSlow o;
    o.n = n;
    o.mean = __ddiv_rn(zs_coop_sum(buf, n, 0.0, false, lane), (double)n);
    o.sd = sqrt(__ddiv_rn(zs_coop_sum(buf, n, o.mean, true, lane), (double)n));
    return o;
}

// One warp = 32 consecutive samples of one target bin at a time; no shared-memory staging on the fast path, so
// occupancy (and with it the latency hiding of the L2 gathers) is bounded by registers only.
__global__ void __launch_bounds__(ZS_WARPS * 32) wc_zscore_kernel(const ZArgs a) {
    extern __shared__ __align__(16) unsigned char zs_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    const int tile = blockIdx.y;
    if (a.npairs != nullptr && *a.npairs <= a.pair_limit) return;       // the pair kernel handles this pass
    const int s = tile * 32 + lane;                      // < ldb by construction
    double* buf = reinterpret_cast<double*>(zs_raw) + (size_t)warp * a.k;      // slow-path scratch, k doubles per warp
    const double* cp = a.copy + s;
    const size_t ldb = (size_t)a.ldb;
    const int bin_end = min(a.N, (int)(blockIdx.x + 1) * ZS_BINS_PER_CTA);
    for (int i = blockIdx.x * ZS_BINS_PER_CTA + warp; i < bin_end; i += nwarps) {
        const int cnt = a.count[i];
        const int* tab = a.table + (size_t)i * a.k;      // every lane reads the same entries: one broadcast sector
        unsigned worst = 0;
        int n = cnt;
        const double sum = zs_stream_sum<false>(cp, tab, cnt, ldb, 0.0, worst);
        double mean = __ddiv_rn(sum, (double)cnt);                          // np_mean (wisetools.py:426)
        double sd = 0.0;
        const bool bad = worst >= 0x7ff00000u;
        if (!bad) {
            unsigned unused = 0;
            sd = sqrt(__ddiv_rn(zs_stream_sum<true>(cp, tab, cnt, ldb, mean, unused), (double)cnt));   // np_std (:427)
        }
        unsigned todo = __ballot_sync(0xffffffffu, bad);
        while (todo) {                                    // warp-uniform loop over the lanes that need the exact compaction
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const ZsSlow o = zs_slow_lane(a.copy + tile * 32 + src, tab, cnt, ldb, buf, lane);
            if (lane == src) { mean = o.mean; sd = o.sd; n = o.n; }
        }
        const double x = a.test[(size_t)i * ldb + s];
        const size_t o = (size_t)i * ldb + s;
        a.z[o] = __ddiv_rn(__dsub_rn(x, mean), sd);                          // wisetools.py:431
        a.r[o] = __ddiv_rn(x, mean);                                         // wisetools.py:432
        a.refsz[o] = n;
        a.sd[o] = sd;
    }
}

// Later passes only touch what changed.  A (bin, sample) pair's statistics depend on the working copy at the bin's
// reference bins only, so after a pass has marked some bins (testCopy[abs(z) >= threshold] = -1, wisetools.py:446) the
// next pass differs from it exactly at the pairs (i, s) with a newly marked j among i's reference bins - everything
// else would be recomputed to the same bits.  wc_mark_kernel applies the marks and raises a dirty flag on those pairs
// through the reverse table; wc_compact_kernel turns the flags into a work list; wc_zscore_pairs_kernel recomputes the
// listed pairs (one pair per lane; gathers are no longer coalesced, but the list is a few per cent of a full pass).
__global__ void wc_mark_kernel(const double* __restrict__ z, double* __restrict__ copy, int N, int B, int ldb, double thr,
                               const int* __restrict__ rev_off, const int* __restrict__ rev_idx,
                               unsigned char* __restrict__ dirty) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)N * ldb) return;
    const int s = (int)(idx % ldb), j = (int)(idx / ldb);
    if (s < B && fabs(z[idx]) >= thr && copy[idx] != -1.0) {      // NaN never marks
        copy[idx] = -1.0;
        for (int e = rev_off[j]; e < rev_off[j + 1]; ++e) dirty[(size_t)rev_idx[e] * ldb + s] = 1;
    }
}

__global__ void wc_compact_kernel(unsigned char* __restrict__ dirty, size_t total, int* __restrict__ pairs,
                                  int* __restrict__ npairs) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool d = idx < total && dirty[idx] != 0;
    if (d) dirty[idx] = 0;                                        // clean for the next pass
    const unsigned bal = __ballot_sync(0xffffffffu, d);
    if (bal == 0) return;
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == 0) base = atomicAdd(npairs, __popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (d) pairs[base + __popc(bal & ((1u << lane) - 1u))] = (int)idx;
}

__global__ void __launch_bounds__(ZS_WARPS * 32) wc_zscore_pairs_kernel(const ZArgs a, const int* __restrict__ pairs,
                                                                        const int* __restrict__ npairs) {
    extern __shared__ __align__(16) unsigned char zs_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    double* buf = reinterpret_cast<double*>(zs_raw) + (size_t)warp * a.k;
    const size_t ldb = (size_t)a.ldb;
    const int n_pairs = *npairs;
    if (n_pairs > a.pair_limit) return;                   // too many for scattered gathers: the full kernel runs instead
    for (int base = (blockIdx.x * nwarps + warp) * 32; base < n_pairs; base += gridDim.x * nwarps * 32) {
        const bool valid = base + lane < n_pairs;
        const int code = valid ? pairs[base + lane] : 0;
        const int i = code / a.ldb, s = code - i * a.ldb;
        const int cnt = valid ? a.count[i] : 0;
        const int* tab = a.table + (size_t)i * a.k;
        const double* cp = a.copy + s;
        unsigned worst = 0;
        int n = cnt;
        double mean = 0.0, sd = 0.0;
        if (valid) {
            mean = __ddiv_rn(zs_stream_sum<false>(cp, tab, cnt, ldb, 0.0, worst), (double)cnt);
            if (worst < 0x7ff00000u) {
                unsigned unused = 0;
                sd = sqrt(__ddiv_rn(zs_stream_sum<true>(cp, tab, cnt, ldb, mean, unused), (double)cnt));
            }
        }
        unsigned todo = __ballot_sync(0xffffffffu, valid && worst >= 0x7ff00000u);
        while (todo) {                                    // warp-cooperative exact compaction, one listed pair at a time
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const int si = __shfl_sync(0xffffffffu, i, src), ss = __shfl_sync(0xffffffffu, s, src);
            const ZsSlow o = zs_slow_lane(a.copy + ss, a.table + (size_t)si * a.k, a.count[si], ldb, buf, lane);
            if (lane == src) { mean = o.mean; sd = o.sd; n = o.n; }
        }
        if (valid) {
            const size_t o = (size_t)i * ldb + s;
            const double x = a.test[o];
            a.z[o] = __ddiv_rn(__dsub_rn(x, mean), sd);
            a.r[o] = __ddiv_rn(x, mean);
            a.refsz[o] = n;
            a.sd[o] = sd;
        }
    }
}

// ---- K8w: the same passes for k > 512 ---------------------------------------------------------------------------
// K8's fast path unrolls numpy's split tree to three levels and its slow path keeps k doubles per warp in shared memory,
// which bounds it at 512.  Here every lane evaluates the split tree over its own kept values in one streaming walk
// (NpStream), so the cost per value is constant and nothing is staged.  The layout is K8's: in the full kernel a warp
// is 32 samples x one bin, the lanes walk the bin's table row in lockstep (a broadcast index load, one coalesced 256 B
// gather per reference bin) and differ only in which values they push.  The tree must be that of the kept count,
// which is only known after a walk: the first walk assumes nothing is dropped (tree of `count`); a lane that dropped
// something walks again with the tree of its kept count.  Then one more walk for sum((x - mean)^2).
template <bool DEV>
__device__ __forceinline__ double zw_walk(const double* cp, const int* tab, int cnt, size_t ldb, int n_tree, double mean,
                                          int& kept) {
    NpStream acc;
    acc.begin(n_tree);
    int nk = 0;
    auto feed = [&](double v) {
        if (v >= 0.0) {                                   // refData[refData >= 0] (wisetools.py:425): NaN never passes
            ++nk;
            if (DEV) {
                const double d = __dsub_rn(v, mean);
                v = __dmul_rn(d, d);
            }
            acc.push(v);
        }
    };
    int m = 0;
    for (; m + 8 <= cnt; m += 8) {
        const int4 i0 = *reinterpret_cast<const int4*>(tab + m), i1 = *reinterpret_cast<const int4*>(tab + m + 4);
        double v[8];
        v[0] = cp[(size_t)i0.x * ldb]; v[1] = cp[(size_t)i0.y * ldb]; v[2] = cp[(size_t)i0.z * ldb]; v[3] = cp[(size_t)i0.w * ldb];
        v[4] = cp[(size_t)i1.x * ldb]; v[5] = cp[(size_t)i1.y * ldb]; v[6] = cp[(size_t)i1.z * ldb]; v[7] = cp[(size_t)i1.w * ldb];
#pragma unroll
        for (int j = 0; j < 8; ++j) feed(v[j]);
    }
    for (; m < cnt; ++m) feed(cp[(size_t)tab[m] * ldb]);
    kept = nk;
    return acc.res;                                       // numpy's sum iff nk == n_tree
}

__device__ __forceinline__ ZsSlow zw_lane(const double* cp, const int* tab, int cnt, size_t ldb) {
    ZsSlow o;
    double sum;
    int n_tree = cnt;
    for (;;) {                                            // at most twice: the second walk uses the kept count
        sum = zw_walk<false>(cp, tab, cnt, ldb, n_tree, 0.0, o.n);
        if (o.n == n_tree) break;
        n_tree = o.n;
    }
    o.mean = __ddiv_rn(sum, (double)o.n);                                                       // np_mean (:426)
    int unused;
    o.sd = sqrt(__ddiv_rn(zw_walk<true>(cp, tab, cnt, ldb, o.n, o.mean, unused), (double)o.n));   // np_std (:427)
    return o;
}

__device__ __forceinline__ void zw_store(const ZArgs& a, int i, int s, const ZsSlow& o) {
    const size_t idx = (size_t)i * a.ldb + s;
    const double x = a.test[idx];
    a.z[idx] = __ddiv_rn(__dsub_rn(x, o.mean), o.sd);                                          // wisetools.py:431
    a.r[idx] = __ddiv_rn(x, o.mean);                                                           // wisetools.py:432
    a.refsz[idx] = o.n;
    a.sd[idx] = o.sd;
}

__global__ void __launch_bounds__(ZS_WARPS * 32) wc_zscore_wide_kernel(const ZArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    if (a.npairs != nullptr && *a.npairs <= a.pair_limit) return;       // the pair kernel handles this pass
    const int s = blockIdx.y * 32 + lane;                // < ldb by construction
    const int bin_end = min(a.N, (int)(blockIdx.x + 1) * ZS_BINS_PER_CTA);
    for (int i = blockIdx.x * ZS_BINS_PER_CTA + warp; i < bin_end; i += nwarps)
        zw_store(a, i, s, zw_lane(a.copy + s, a.table + (size_t)i * a.k, a.count[i], (size_t)a.ldb));
}

// Dirty-pair pass for k > 512: one listed pair per thread, the same walk as the full kernel.
__global__ void __launch_bounds__(ZS_WARPS * 32) wc_zscore_wide_pairs_kernel(const ZArgs a, const int* __restrict__ pairs,
                                                                             const int* __restrict__ npairs) {
    const int n_pairs = *npairs;
    if (n_pairs > a.pair_limit) return;                   // too many for scattered gathers: the full kernel runs instead
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n_pairs; e += gridDim.x * blockDim.x) {
        const int code = pairs[e];
        const int i = code / a.ldb, s = code - i * a.ldb;
        zw_store(a, i, s, zw_lane(a.copy + s, a.table + (size_t)i * a.k, a.count[i], (size_t)a.ldb));
    }
}

// stdDevSum / stdDevNum accumulated bin by bin like the reference's Python loop (wisetools.py:428-430, 435): a strictly
// sequential sum per sample, so the parallelism is across samples only.  A CTA owns 32 samples: all eight warps stream
// the [64 bins][32 samples] tiles of the sigma array into shared memory (coalesced, cp.async, double buffered) and warp 0
// - one lane per sample - walks each tile in bin order.
constexpr int SG_BINS = 64;    // 2 x 64 x 32 doubles = 32 KB of static shared memory
__global__ void __launch_bounds__(256) wc_sigma_kernel(const double* __restrict__ sd, int N, int B, int ldb,
                                                       double* __restrict__ asdef) {
    __shared__ double tile[2][SG_BINS][32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s0 = blockIdx.x * 32;
    auto issue = [&](int chunk, int buf) {
        const int b0 = chunk * SG_BINS;
        for (int e = tid; e < SG_BINS * 32; e += 256) {
            const int bin = e >> 5, l = e & 31;
            if (b0 + bin < N) zs_cp_async_8(&tile[buf][bin][l], sd + (size_t)(b0 + bin) * ldb + s0 + l);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    const int nchunks = (N + SG_BINS - 1) / SG_BINS;
    double sum = 0.0;
    int num = 0;
    issue(0, 0);
    for (int c = 0; c < nchunks; ++c) {
        if (c + 1 < nchunks) {
            issue(c + 1, (c + 1) & 1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        if (warp == 0) {
            const int nb = min(SG_BINS, N - c * SG_BINS);
            const double* col = &tile[c & 1][0][lane];
#pragma unroll 8
            for (int bin = 0; bin < nb; ++bin) {
                // a skipped bin adds +0.0 (sum >= +0 throughout: the same bits as not adding): the select sits before the
                // add, so the loop-carried chain is one DADD per bin
                const double v = col[bin * 32];
                const bool ok = !isnan(v);
                sum = __dadd_rn(sum, ok ? v : 0.0);
                num += ok ? 1 : 0;
            }
        }
        __syncthreads();
    }
    if (warp == 0 && s0 + lane < B) asdef[s0 + lane] = __ddiv_rn(sum, (double)num);
}

// [N][ldb] sample-minor -> [B][N] sample-major (what the host copies out and what the segmentation reads)
template <class T>
__global__ void wc_transpose_kernel(const T* __restrict__ in, int N, int B, int ldb, T* __restrict__ out) {
    __shared__ T tile[32][33];
    const int n0 = blockIdx.x * 32, b0 = blockIdx.y * 32;
    {
        const int n = n0 + threadIdx.y, b = b0 + threadIdx.x;
        if (n < N && b < ldb) tile[threadIdx.y][threadIdx.x] = in[(size_t)n * ldb + b];
    }
    __syncthreads();
    const int n = n0 + threadIdx.x, b = b0 + threadIdx.y;
    if (n < N && b < B) out[(size_t)b * N + n] = tile[threadIdx.x][threadIdx.y];
}

int upload_row_ranges(wc_ctx* ctx, int N, const int* chrom_bins_h, int nchrom, int slot_cs, int slot_ce, int** cs_d,
                      int** ce_d, cudaStream_t stream) {
    std::vector<int> row_cs(N), row_ce(N);
    int pos = 0;
    for (int c = 0; c < nchrom; ++c) {
        for (int i = 0; i < chrom_bins_h[c]; ++i) { row_cs[pos + i] = pos; row_ce[pos + i] = pos + chrom_bins_h[c]; }
        pos += chrom_bins_h[c];
    }
    int rc;
    ctx->sched_hash = 0;                         // these slots are shared with the search: its cached metadata is gone
    if ((rc = wc_reserve(ctx, slot_cs, (size_t)N * sizeof(int), (void**)cs_d))) return rc;
    if ((rc = wc_reserve(ctx, slot_ce, (size_t)N * sizeof(int), (void**)ce_d))) return rc;
    WC_CUDA(cudaMemcpyAsync(*cs_d, row_cs.data(), (size_t)N * sizeof(int), cudaMemcpyHostToDevice, stream));
    WC_CUDA(cudaMemcpyAsync(*ce_d, row_ce.data(), (size_t)N * sizeof(int), cudaMemcpyHostToDevice, stream));
    WC_CUDA(cudaStreamSynchronize(stream));      // the host vectors die with this frame
    return WC_OK;
}

}  // namespace

extern "C" int wc_table_stride(int k) { return (k + 3) & ~3; }

// The table, the reverse table and the dirty-pair codes are indexed with int32: N x wc_table_stride(k) must stay below
// 2^31 (k <= 37 260 at 50 kb, N = 57 633; k <= 7 452 at 10 kb).  Checked before any memory is touched.
static int check_table_size(int N, int k) {
    const long long stride = ((long long)k + 3) & ~3LL;
    if ((long long)N * stride >= (1LL << 31)) {
        wc_set_error("bad argument: N x wc_table_stride(k) = %d x %lld must be below 2^31 (refsize too large for %d bins)",
                     N, stride, N);
        return WC_ERR_ARG;
    }
    return WC_OK;
}

extern "C" int wc_test_table(wc_ctx* ctx, const int32_t* indexes_d, const double* distances_d, int N, int k,
                             const int* chrom_bins_h, int nchrom, double cutoff, int32_t* table_d, int32_t* count_d,
                             int32_t* rev_off_d, int32_t* rev_idx_d, void* stream_v) {
    WC_CHECK_ARG(ctx != nullptr && indexes_d != nullptr && distances_d != nullptr && chrom_bins_h != nullptr);
    WC_CHECK_ARG(table_d != nullptr && count_d != nullptr && rev_off_d != nullptr && rev_idx_d != nullptr);
    WC_CHECK_ARG(N > 0 && k > 0 && nchrom > 0);
    long long tot = 0;
    for (int c = 0; c < nchrom; ++c) { WC_CHECK_ARG(chrom_bins_h[c] >= 0); tot += chrom_bins_h[c]; }
    WC_CHECK_ARG(tot == N);
    int rc;
    if ((rc = check_table_size(N, k))) return rc;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    WC_CUDA(cudaSetDevice(ctx->device));
    int* cs_d; int* ce_d;
    if ((rc = upload_row_ranges(ctx, N, chrom_bins_h, nchrom, SLOT_ROWCS, SLOT_ROWCE, &cs_d, &ce_d, stream))) return rc;
    const int blocks = (int)(((size_t)N * 32 + 255) / 256);
    const int ldk = wc_table_stride(k);
    wc_table_kernel<<<blocks, 256, 0, stream>>>(indexes_d, distances_d, N, k, ldk, cs_d, ce_d, cutoff, table_d, count_d);
    // reverse table (CSR): counting sort of the (bin -> reference bin) edges by reference bin
    int* rev_cnt; int* cursor;
    if ((rc = wc_reserve(ctx, SLOT_T_REVCNT, (size_t)N * sizeof(int), (void**)&rev_cnt))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_T_REVCUR, (size_t)N * sizeof(int), (void**)&cursor))) return rc;
    WC_CUDA(cudaMemsetAsync(rev_cnt, 0, (size_t)N * sizeof(int), stream));
    wc_rev_count_kernel<<<blocks, 256, 0, stream>>>(table_d, count_d, N, ldk, rev_cnt);
    wc_rev_scan_kernel<<<1, 1024, 0, stream>>>(rev_cnt, N, rev_off_d, cursor);
    wc_rev_fill_kernel<<<blocks, 256, 0, stream>>>(table_d, count_d, N, ldk, cursor, rev_idx_d);
    WC_CUDA(cudaGetLastError());
    return WC_OK;
}

template <class TIn>
static int prep_common(wc_ctx* ctx, const TIn* in_d, int ld_in, const int* map_d, bool normalise, int B, int N,
                       const double* pca_mean_d, const double* pca_components_d, int ncomp, double* test_d, int ldb,
                       cudaStream_t stream) {
    double* totals = nullptr; double* proj;
    int rc;
    if ((rc = wc_reserve(ctx, SLOT_T_PROJ, (size_t)B * std::max(ncomp, 1) * sizeof(double), (void**)&proj))) return rc;
    WC_CUDA(cudaEventRecord(ctx->ev[12], stream));
    if (normalise) {
        if ((rc = wc_reserve(ctx, SLOT_T_TOTALS, (size_t)B * sizeof(double), (void**)&totals))) return rc;
        wc_totals_kernel<<<B, 256, 0, stream>>>(reinterpret_cast<const int*>(in_d), ld_in, totals);
    }
    if (ncomp > 0)
        wc_project_kernel<TIn><<<B, 256, 0, stream>>>(in_d, ld_in, map_d, N, totals, pca_mean_d, pca_components_d, ncomp, proj);
    dim3 grid((N + 31) / 32, ldb / 32);
    wc_residual_kernel<TIn><<<grid, dim3(32, 32), 0, stream>>>(in_d, ld_in, map_d, N, B, ldb, totals, pca_mean_d,
                                                               pca_components_d, ncomp, proj, test_d);
    WC_CUDA(cudaGetLastError());
    WC_CUDA(cudaEventRecord(ctx->ev[13], stream));
    ctx->timed_mask |= 1u << 6;
    return WC_OK;
}

extern "C" int wc_test_prep(wc_ctx* ctx, const int32_t* counts_d, int B, int Nraw, const int32_t* masked_raw_d, int N,
                            const double* pca_mean_d, const double* pca_components_d, int ncomp, double* test_d, int ldb,
                            void* stream_v) {
    WC_CHECK_ARG(ctx != nullptr && counts_d != nullptr && masked_raw_d != nullptr && test_d != nullptr);
    WC_CHECK_ARG(ncomp == 0 || (pca_mean_d != nullptr && pca_components_d != nullptr));
    WC_CHECK_ARG(B > 0 && Nraw > 0 && N > 0 && N <= Nraw && ncomp >= 0 && ldb >= B && ldb % 32 == 0);
    WC_CUDA(cudaSetDevice(ctx->device));
    return prep_common<int>(ctx, counts_d, Nraw, masked_raw_d, true, B, N, pca_mean_d, pca_components_d, ncomp, test_d,
                            ldb, static_cast<cudaStream_t>(stream_v));
}

extern "C" int wc_apply_pca(wc_ctx* ctx, const double* x_d, int B, int N, const double* pca_mean_d,
                            const double* pca_components_d, int ncomp, double* test_d, int ldb, void* stream_v) {
    WC_CHECK_ARG(ctx != nullptr && x_d != nullptr && test_d != nullptr && pca_mean_d != nullptr && pca_components_d != nullptr);
    WC_CHECK_ARG(B > 0 && N > 0 && ncomp > 0 && ldb >= B && ldb % 32 == 0);
    WC_CUDA(cudaSetDevice(ctx->device));
    return prep_common<double>(ctx, x_d, N, nullptr, false, B, N, pca_mean_d, pca_components_d, ncomp, test_d, ldb,
                               static_cast<cudaStream_t>(stream_v));
}

extern "C" int wc_zscore_batch(wc_ctx* ctx, const double* test_d, const double* copy_init_d, int N, int B, int ldb,
                               const int32_t* table_d, const int32_t* count_d, const int32_t* rev_off_d,
                               const int32_t* rev_idx_d, int k, double z_threshold, int repeats, double* z_d, double* r_d,
                               int32_t* refsizes_d, double* asdef_d, void* stream_v) {
    WC_CHECK_ARG(ctx != nullptr && test_d != nullptr && table_d != nullptr && count_d != nullptr);
    WC_CHECK_ARG(z_d != nullptr && r_d != nullptr && refsizes_d != nullptr && asdef_d != nullptr);
    WC_CHECK_ARG(N > 0 && B > 0 && ldb >= B && ldb % 32 == 0 && k >= 1 && repeats >= 1);
    WC_CHECK_ARG(repeats == 1 || (rev_off_d != nullptr && rev_idx_d != nullptr));
    WC_CHECK_ARG((size_t)N * ldb < ((size_t)1 << 31));
    int rc;
    if ((rc = check_table_size(N, k))) return rc;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    WC_CUDA(cudaSetDevice(ctx->device));
    const size_t elems = (size_t)N * ldb;
    double* copy; double* zt; double* rt; int* nt; double* sd; unsigned char* dirty; int* pairs; int* npairs;
    if ((rc = wc_reserve(ctx, SLOT_T_COPY, elems * sizeof(double), (void**)&copy))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_T_ZT, elems * sizeof(double), (void**)&zt))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_T_RT, elems * sizeof(double), (void**)&rt))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_T_NT, elems * sizeof(int), (void**)&nt))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_T_SD, elems * sizeof(double), (void**)&sd))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_T_FLAGS, (size_t)(repeats + 1) * sizeof(int), (void**)&npairs))) return rc;
    WC_CUDA(cudaEventRecord(ctx->ev[8], stream));
    WC_CUDA(cudaMemcpyAsync(copy, copy_init_d ? copy_init_d : test_d, elems * sizeof(double), cudaMemcpyDeviceToDevice,
                            stream));                                                                   // wisetools.py:442
    const int warps = ZS_WARPS;
    const int ldk = wc_table_stride(k);
    const bool wide = k > 512;                  // K8's sums and slow-path scratch stop at 512 values: K8w beyond
    const size_t smem = wide ? 0 : (size_t)warps * ldk * sizeof(double);     // slow-path scratch only
    if (!wide) {
        WC_CUDA(cudaFuncSetAttribute(wc_zscore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        WC_CUDA(cudaFuncSetAttribute(wc_zscore_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    ZArgs a;
    a.test = test_d; a.copy = copy; a.table = table_d; a.count = count_d; a.N = N; a.B = B; a.ldb = ldb; a.k = ldk;
    a.z = zt; a.r = rt; a.refsz = nt; a.sd = sd; a.npairs = nullptr;
    // a listed pair gathers with 32-byte sectors for 8 useful bytes and shares nothing with its warp: past ~1/8 of all
    // pairs a full coalesced pass is cheaper
    a.pair_limit = (int)std::min<size_t>((size_t)N * B / 8, (size_t)0x7fffffff);
    long long launches = 0;
    const dim3 zgrid((N + ZS_BINS_PER_CTA - 1) / ZS_BINS_PER_CTA, ldb / 32);
    if (wide) wc_zscore_wide_kernel<<<zgrid, warps * 32, 0, stream>>>(a);
    else wc_zscore_kernel<<<zgrid, warps * 32, smem, stream>>>(a);       // first pass: every (bin, sample) pair
    ++launches;
    if (repeats > 1) {
        if ((rc = wc_reserve(ctx, SLOT_T_DIRTY, elems, (void**)&dirty))) return rc;
        if ((rc = wc_reserve(ctx, SLOT_T_PAIRS, elems * sizeof(int), (void**)&pairs))) return rc;
        WC_CUDA(cudaMemsetAsync(dirty, 0, elems, stream));
        WC_CUDA(cudaMemsetAsync(npairs, 0, (size_t)(repeats + 1) * sizeof(int), stream));
        const unsigned eblocks = (unsigned)((elems + 255) / 256);
        for (int rep = 1; rep < repeats; ++rep) {     // the marks of the last pass are never read (wisetools.py:443-448)
            wc_mark_kernel<<<eblocks, 256, 0, stream>>>(zt, copy, N, B, ldb, z_threshold, rev_off_d, rev_idx_d, dirty);
            wc_compact_kernel<<<eblocks, 256, 0, stream>>>(dirty, elems, pairs, npairs + rep);
            a.npairs = npairs + rep;                   // exactly one of the next two kernels does the pass
            if (wide) {
                wc_zscore_wide_pairs_kernel<<<4 * ctx->sm_count, warps * 32, 0, stream>>>(a, pairs, npairs + rep);
                wc_zscore_wide_kernel<<<zgrid, warps * 32, 0, stream>>>(a);
            } else {
                wc_zscore_pairs_kernel<<<4 * ctx->sm_count, warps * 32, smem, stream>>>(a, pairs, npairs + rep);
                wc_zscore_kernel<<<zgrid, warps * 32, smem, stream>>>(a);
            }
            launches += 4;
        }
    }
    wc_sigma_kernel<<<ldb / 32, 256, 0, stream>>>(sd, N, B, ldb, asdef_d);
    dim3 tgrid((N + 31) / 32, ldb / 32);
    wc_transpose_kernel<double><<<tgrid, dim3(32, 32), 0, stream>>>(zt, N, B, ldb, z_d);
    wc_transpose_kernel<double><<<tgrid, dim3(32, 32), 0, stream>>>(rt, N, B, ldb, r_d);
    wc_transpose_kernel<int><<<tgrid, dim3(32, 32), 0, stream>>>(nt, N, B, ldb, refsizes_d);
    launches += 4;
    WC_CUDA(cudaGetLastError());
    WC_CUDA(cudaEventRecord(ctx->ev[9], stream));
    ctx->timed_mask |= 1u << 4;
    ctx->counter[5] = launches;
    ctx->zs_npairs_d = repeats > 1 ? npairs : nullptr;
    ctx->zs_repeats = repeats;
    ctx->zs_pair_limit = a.pair_limit;
    ctx->zs_all_pairs = (long long)N * B;
    return WC_OK;
}
