// wisecondor_b200 - Stouffer segmentation of the z-scores on B200 (sm_100a).
//
// Replaces fillTri + TriArr.segmentTri (/root/reference/wisetools.py:466-472, /root/reference/triarray.py:59-84) and
// the chromosome loop of toolTest (/root/reference/wisecondor.py:233-238) for a batch of samples: per (sample,
// chromosome) the z-scores of the kept bins are compacted, every contiguous run [x..y] is scored
// sum(z[x..y]) / sqrt(y-x+1), the most significant run above the threshold is called and the search recurses to its
// left and right.  The reference materialises the n(n+1)/2 run values (99 MB for chr1 at 50 kb) with an O(n) numpy sum
// each; here one CTA keeps the chromosome's prefix sums in shared memory and sweeps the triangle by diagonals (run lengths)
// with the 1/sqrt(len) factors in registers.
//
// Exactness.  The sweep scores runs from prefix-sum differences times 1/sqrt(len) - not numpy's summation order - so it
// is used only to *locate*, and it tracks one number: M = max |score|.  (The reference takes the maximum, then the
// minimum, and prefers the minimum iff abs(min) > max, triarray.py:62-70: that is always the run of largest |score|,
// the positive one on an exact tie.)  Every run whose |score| lies within a rigorous error window `delta` of M is
// re-scored in numpy's own pairwise order (wc_numpy_order.cuh) and divided by sqrt(len) exactly as the reference does;
// the max / min / abs rule and first-occurrence tie-breaking (the reference's row-major triangle order: smallest x,
// then smallest y) are decided on those exact values.  Calls and their z are identical to the reference's.
//
// K9 wc_segment_kernel   one CTA per (sample, chromosome): compaction -> prefix sums -> [sweep -> exact re-score of the
//                        windowed rows -> call -> push left/right ranges]*                       (FP64 ALU / shared memory)
#include "wc_common.cuh"
#include "wc_numpy_order.cuh"

namespace {

constexpr int SEG_THREADS = 128;
constexpr int SEG_WARPS = SEG_THREADS / 32;
constexpr int SEG_R = 5;                      // run lengths per lane in the sweep (odd: conflict-free prefix reads)
constexpr int SEG_TILE = 32 * SEG_R;          // run lengths per warp tile
constexpr int SEG_ROWCAP = 1024;              // diagonals re-scored exactly per search before falling back to all of them
constexpr double SEG_EPS = 1.1102230246251565e-16;
constexpr double SEG_FLT_TINY = 8.0 * 1.1754943508222875e-38;   // 8 x FLT_MIN: flush / subnormal rounding of the fp32 sweep

struct SegArgs {
    const double* z;         // [B][N]
    const int* refsz;        // [B][N]
    int N, B;
    const int* sel_start;    // [nsel] first masked bin of each selected chromosome (sorted by descending length)
    const int* sel_len;      // [nsel]
    const int* sel_slot;     // [nsel] position of the chromosome in the caller's list
    const int* sel_soff;     // [nsel] global stack: entries of the selected chromosomes before this one, per sample
    int nsel;
    int minrefbins;
    double thr;
    int min_search;
    double* zc;              // [B][N] scratch: kept z-scores of (sample, chromosome) compacted at the chromosome's offset
    const double* r;         // [B][N] ratios (resultsR); only for the effect-size filter
    double* rc;              // [B][N] scratch: kept ratios, compacted like zc
    double c_hi, c_lo;       // fillTriMin keeps a run iff median(R) >= c_hi or median(R) <= c_lo (= abs(median - 1) >= t)
    double* cwz;             // [B][nsel]
    int* cleaned;            // [B][nsel]
    wc_call* calls;          // [B][max_calls]
    int* ncalls;             // [B]
    int max_calls;
    int pcap;                // capacity of the per-chromosome arrays (>= longest chromosome + 1)
    unsigned* aux_g;         // when the side arrays do not fit in shared memory next to P: [blocks][pcap * aux_words] global
    int* stack_g;            // when the stack does not fit in shared memory: per (chromosome, sample) 2 * scap ints, scap
                             // from that chromosome's length (else in shared memory after P / aux, sized for the longest)
    int* status;             // [0] |= 1 call overflow, 2 range-stack overflow, 4 |z| sums beyond 2^1023, 8 empty window
};

struct Best {                // lexicographic champion: value, then first occurrence (x, then y)
    double v;
    int x, y;
};
__device__ __forceinline__ bool better_max(const Best& a, const Best& b) {   // a beats b
    return a.v > b.v || (a.v == b.v && (a.x < b.x || (a.x == b.x && a.y < b.y)));
}
__device__ __forceinline__ bool better_min(const Best& a, const Best& b) {
    return a.v < b.v || (a.v == b.v && (a.x < b.x || (a.x == b.x && a.y < b.y)));
}
__device__ __forceinline__ Best shfl_best(const Best& b, int o) {
    Best r;
    r.v = __shfl_xor_sync(0xffffffffu, b.v, o);
    r.x = __shfl_xor_sync(0xffffffffu, b.x, o);
    r.y = __shfl_xor_sync(0xffffffffu, b.y, o);
    return r;
}

// MINEFF: fillTriMin's effect-size filter (wisetools.py:475-487): a run only counts if abs(median(R[x..y]) - 1) >=
// mineffectsize, otherwise its triangle entry is 0 (and 0 never wins against a positive threshold).
template <bool MINEFF>
__global__ void __launch_bounds__(SEG_THREADS) wc_segment_kernel(const SegArgs a) {
    extern __shared__ __align__(16) unsigned char seg_raw[];
    float* P = reinterpret_cast<float*>(seg_raw);                 // [pcap] prefix sums (fp32 copy), P[i] = sum zc[0..i)
    // side arrays: in shared memory after P when they fit, else a per-CTA slice of global scratch
    float* dh = a.aux_g ? reinterpret_cast<float*>(a.aux_g + (size_t)blockIdx.x * a.pcap * (MINEFF ? 4 : 1))
                        : P + a.pcap;                             // [pcap] per run length: max |score| of the sweep
    int* CH = reinterpret_cast<int*>(dh + a.pcap);                // [pcap] MINEFF: #{j < i : rc[j] >= c_hi}
    int* CL = CH + a.pcap;                                        // [pcap] MINEFF: #{j < i : rc[j] <= c_lo}
    int* CN = CL + a.pcap;                                        // [pcap] MINEFF: #{j < i : rc[j] is NaN} (only if there is one)
    __shared__ double s_red[2][SEG_WARPS];
    __shared__ Best s_best[2][SEG_WARPS];
    __shared__ int s_scan[SEG_WARPS];
    __shared__ int s_cur[2];                     // the range popped by thread 0
    __shared__ int s_rows[SEG_ROWCAP];
    __shared__ int s_nrows, s_sp, s_n, s_bad, s_rnan;
    __shared__ unsigned long long s_cand[3];     // MINEFF: first passing NaN / +inf / -inf entry of a range, (x << 32) | y
    __shared__ double s_A, s_Pm, s_scale;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sel = blockIdx.x / a.B, b = blockIdx.x % a.B;     // long chromosomes first
    const int cstart = a.sel_start[sel], clen = a.sel_len[sel], slot = a.sel_slot[sel];
    const double* zrow = a.z + (size_t)b * a.N + cstart;
    const int* nrow = a.refsz + (size_t)b * a.N + cstart;
    double* zc = a.zc + (size_t)b * a.N + cstart;                 // kept z-scores of this chromosome (global scratch)
    double* rc = MINEFF ? a.rc + (size_t)b * a.N + cstart : nullptr;
    const double* rrow = MINEFF ? a.r + (size_t)b * a.N + cstart : nullptr;
    // pending ranges (lo, hi): disjoint and longer than min_search (triarray.py:76-82), so at most
    // clen / (min_search + 1) + 1 are ever pending.  In shared memory after the side arrays when they fit, else a slice
    // of global scratch sized for this chromosome.
    const int scap = clen / (a.min_search + 1) + 1;
    int* stk = a.stack_g ? a.stack_g + 2 * ((size_t)a.sel_soff[sel] * a.B + (size_t)b * scap)
                         : reinterpret_cast<int*>(a.aux_g ? P + a.pcap : dh + (size_t)a.pcap * (MINEFF ? 4 : 1));

    // ---- 1. compaction of the kept bins (wisecondor.py:215-218: refSizes >= minrefbins) -------------------------
    if (tid == 0) { s_n = 0; s_bad = 0; s_rnan = 0; }
    __syncthreads();
    for (int base = 0; base < clen; base += SEG_THREADS) {
        const int i = base + tid;
        const bool keep = i < clen && nrow[i] >= a.minrefbins;
        const double v = keep ? zrow[i] : 0.0;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_scan[warp] = __popc(bal);
        __syncthreads();
        int off = s_n;
        for (int w = 0; w < warp; ++w) off += s_scan[w];
        if (keep) {
            zc[off + __popc(bal & ((1u << lane) - 1u))] = v;
            if (MINEFF) {
                const double rv = rrow[i];
                rc[off + __popc(bal & ((1u << lane) - 1u))] = rv;
                if (isnan(rv)) s_rnan = 1;
            }
            if (!isfinite(v)) s_bad = 1;
        }
        __syncthreads();
        if (tid == 0) {
            int t = 0;
            for (int w = 0; w < SEG_WARPS; ++w) t += s_scan[w];
            s_n += t;
        }
        __syncthreads();
    }
    const int n = s_n;                              // (the __syncthreads above also orders the global zc writes)
    if (tid == 0) a.cleaned[(size_t)b * a.nsel + slot] = n;
    if (n == 0) {                                   // the reference raises on an empty chromosome (triarray.py:29)
        if (tid == 0) a.cwz[(size_t)b * a.nsel + slot] = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }
    // +-inf / NaN z (a kept bin whose reference sigma is 0, wisetools.py:431 under np.seterr('ignore')): the reference's
    // argmax/argmin then see inf / NaN run values; handled per range below.  Prefix sums skip the non-finite bins.
    const bool has_bad = s_bad != 0;
    // A NaN ratio (0 / 0: an empty bin whose reference bins are empty too) makes np_median of every run that holds it NaN
    // and the filter's comparison False (wisetools.py:483): such runs are zeroed.  +-inf ratios order like any value.
    const bool has_rnan = MINEFF && s_rnan != 0;

    // ---- 2. prefix sums and A = sum |z| (the scale of the error window) ---------------------------------------------
    {
        const int per = (n + SEG_THREADS - 1) / SEG_THREADS;
        const int i0 = min(n, tid * per), i1 = min(n, i0 + per);
        double loc = 0.0, la = 0.0;
        for (int i = i0; i < i1; ++i) {
            const double v = zc[i];
            if (isfinite(v)) { loc += v; la += fabs(v); }
        }
        double inc = loc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) la += __shfl_xor_sync(0xffffffffu, la, o);
        if (lane == 31) s_red[0][warp] = inc;
        if (lane == 0) s_red[1][warp] = la;
        __syncthreads();
        double base = 0.0, at = 0.0;
        for (int w = 0; w < warp; ++w) base += s_red[0][w];
        for (int w = 0; w < SEG_WARPS; ++w) at += s_red[1][w];
        // The fp32 copy is stored x 2^-k so that it never overflows (|P| <= sum |z| = at) and keeps its precision for
        // tiny z: k = 0 unless sum |z| lies outside [2^-60, 2^100], then the scaled sum lies in [2^64, 2^65).  A power of
        // two is exact (short of fp32 underflow, which delta covers), so the sweep, its window and the threshold test
        // all work in scaled units; the exact phase reads the unscaled zc.
        const int k = (at > 0x1p100 || (at > 0.0 && at < 0x1p-60)) && at < 0x1p1023 ? max(ilogb(at) - 64, -1000) : 0;
        const double sc = ldexp(1.0, -k);
        double run = base + (inc - loc);
        double pm = 0.0;                              // largest |prefix sum| (scaled): the scale of the fp32 rounding
        for (int i = i0; i < i1; ++i) {
            const double v = zc[i];
            P[i] = (float)(run * sc);
            pm = fmax(pm, fabs(run * sc));
            if (isfinite(v)) run += v;
        }
        if (i1 == n && i0 < n) { P[n] = (float)(run * sc); pm = fmax(pm, fabs(run * sc)); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) pm = fmax(pm, __shfl_xor_sync(0xffffffffu, pm, o));
        __syncthreads();                              // s_red[0] (warp totals) has been consumed
        if (lane == 0) s_red[0][warp] = pm;
        __syncthreads();
        if (tid == 0) {
            double t = 0.0, m = 0.0;
            for (int w = 0; w < SEG_WARPS; ++w) { t += s_red[1][w]; m = fmax(m, s_red[0][w]); }
            s_A = t;
            s_Pm = m;
            s_scale = sc;
            s_sp = 1;
            stk[0] = 0;
            stk[1] = n;
        }
        __syncthreads();
    }
    // Sums of |z| at or beyond 2^1023 can overflow double precision in numpy's sums (the reference's run values would
    // be inf or NaN); such a chromosome is rejected as a whole (WC_ERR_ARG) instead of being located on non-finite
    // prefix sums.  Below 2^1023 every partial sum in any order is finite.
    if (!(s_A < 0x1p1023)) {
        if (tid == 0) atomicOr(a.status, 4);
        return;
    }
    const double scale = s_scale;                   // 2^-k of the fp32 copy; 1 unless sum |z| is outside [2^-60, 2^100]
    const double thr_s = a.thr * scale;             // the threshold in the sweep's units (inf / 0 when out of range)
    const double A = s_A * scale;
    // |sweep value - numpy value| <= (2 (per + 16) + 40) eps A + 3 eps |v|: prefix sums (sequential chunk of `per`, warp
    // scan, warp bases) on both ends of the run, numpy's own pairwise rounding, the reciprocal multiply.  delta = 2 x that.
    // The sweep itself runs in fp32 on an fp32 copy of the prefix sums: |fp32 score - fp64 score| <= 2^-23 Pm + 2^-21 |v|
    // (rounding of the two prefix sums, of their difference, of 1/sqrt(len) and of the product), Pm = max |prefix sum|.
    // Scaled values that fall below FLT_MIN are flushed or rounded to the subnormal grid: SEG_FLT_TINY bounds that on the
    // two prefix sums, their difference and the product.  All of delta is in the sweep's (scaled) units.
    const double delta_A = (4.0 * ((n + SEG_THREADS - 1) / SEG_THREADS) + 160.0) * SEG_EPS * A + 2.0 * 1.1920929e-07 * s_Pm
                           + SEG_FLT_TINY;

    // MINEFF: prefix counts of the ratios above c_hi / below c_lo decide the median test in O(1) for all odd lengths and
    // for even lengths unless exactly half of the run lies on the far side; then the two middle order statistics are
    // the largest value on the near side and the smallest on the far side (one scan of the run).
    if (MINEFF) {
        if (tid == 0) {
            int ch = 0, cl = 0;
            for (int i = 0; i < n; ++i) {
                CH[i] = ch; CL[i] = cl;
                const double rv = rc[i];
                ch += rv >= a.c_hi ? 1 : 0;
                cl += rv <= a.c_lo ? 1 : 0;
            }
            CH[n] = ch; CL[n] = cl;
        }
        if (has_rnan && tid == 32) {
            int cn = 0;
            for (int i = 0; i < n; ++i) { CN[i] = cn; cn += isnan(rc[i]) ? 1 : 0; }
            CN[n] = cn;
        }
        __syncthreads();
    }
    auto passes = [&](int x, int L) -> bool {          // abs(np_median(regionR[x:y+1]) - 1) >= threshold (wisetools.py:483)
        if (!MINEFF) return true;
        if (has_rnan && CN[x + L] != CN[x]) return false;
        const int mid = L >> 1;
        const int nh = CH[x + L] - CH[x], nl = CL[x + L] - CL[x];
        if (L & 1) return nh >= mid + 1 || nl >= mid + 1;            // the median is the middle element
        if (nh >= mid + 1 || nl >= mid + 1) return true;             // both middle elements on the far side
        bool ok = false;
        if (nh == mid) {                              // a_mid < c_hi <= a_mid+1: median = (a_mid + a_mid+1) / 2
            double below = -INFINITY, above = INFINITY;
            for (int i = x; i < x + L; ++i) {
                const double rv = rc[i];
                if (rv >= a.c_hi) above = fmin(above, rv); else below = fmax(below, rv);
            }
            ok = __ddiv_rn(__dadd_rn(below, above), 2.0) >= a.c_hi;
        }
        if (!ok && nl == mid) {
            double below = -INFINITY, above = INFINITY;
            for (int i = x; i < x + L; ++i) {
                const double rv = rc[i];
                if (rv <= a.c_lo) below = fmax(below, rv); else above = fmin(above, rv);
            }
            ok = __ddiv_rn(__dadd_rn(below, above), 2.0) <= a.c_lo;
        }
        return ok;
    };

    // chromosome-wide value: entry (0, n-1) of the triangle (wisecondor.py:237), numpy order, by one thread (a non-finite
    // bin propagates through the same additions: inf, or NaN for inf - inf)
    if (tid == SEG_THREADS - 1) {
        const double tot = np_sum_thread([&](int i) { return zc[i]; }, n);
        a.cwz[(size_t)b * a.nsel + slot] = passes(0, n) ? __ddiv_rn(tot, sqrt((double)n)) : 0.0;
    }
    __shared__ int s_first[3];                      // first NaN / +inf / -inf position of the current range

    // ---- 3. iterative most-significant-run search (triarray.py:59-84) --------------------------------------------------
    // the stack holds scap ranges (see stk above); status 2 is an internal assertion
    auto push = [&](int spn, int l, int h) -> int {
        if (spn < scap) { stk[2 * spn] = l; stk[2 * spn + 1] = h; return spn + 1; }
        atomicOr(a.status, 2);
        return spn;
    };
    while (true) {
        __syncthreads();
        if (tid == 0) {
            const int sp = s_sp;
            if (sp > 0) { s_cur[0] = stk[2 * (sp - 1)]; s_cur[1] = stk[2 * (sp - 1) + 1]; s_sp = sp - 1; }
            else s_cur[0] = -1;
        }
        __syncthreads();
        const int lo = s_cur[0], hi = s_cur[1];
        if (lo < 0) break;
        const int m = hi - lo;

        if (MINEFF && has_bad) {
            // With the effect-size filter an inf / NaN run only counts where its median test passes (the others are 0):
            // the first NaN entry in row-major order (numpy's argmax / argmin, triarray.py:62-66), else the first +inf
            // entry (the maximum), else the first -inf entry (abs(min) > max, :68-70).  A row's run values go finite ->
            // +-inf -> NaN as y grows; one thread per row x walks y and tests the non-finite stretch (rare path: O(m^2)
            // median tests in all).  No passing non-finite entry: the finite sweep below decides - runs holding a
            // non-finite bin do not pass there either.
            if (tid < 3) s_cand[tid] = ~0ull;
            __syncthreads();
            for (int xb = lo; xb < hi; xb += SEG_THREADS) {
                const int x = xb + tid;
                if (x < hi) {
                    bool sn = false, sp = false, sm = false, gotp = false, gotm = false;
                    for (int y = x; y < hi; ++y) {
                        const double v = zc[y];
                        if (!isfinite(v)) {
                            if (isnan(v)) sn = true; else if (v > 0.0) sp = true; else sm = true;
                        }
                        const int kind = (sn || (sp && sm)) ? 0 : (sp ? 1 : (sm ? 2 : -1));
                        if (kind < 0 || (kind == 1 && gotp) || (kind == 2 && gotm)) continue;
                        if (passes(x, y - x + 1)) {
                            atomicMin(&s_cand[kind], ((unsigned long long)x << 32) | (unsigned)y);
                            if (kind == 0) break;                  // the rest of the row comes later in the order
                            if (kind == 1) gotp = true; else gotm = true;
                        }
                    }
                }
                __syncthreads();
                const bool stop = s_cand[0] != ~0ull;              // a NaN entry in these rows: no later row precedes it
                __syncthreads();
                if (stop) break;
            }
            const unsigned long long cn = s_cand[0], cp = s_cand[1], cm = s_cand[2];
            if ((cn & cp & cm) != ~0ull) {
                __syncthreads();                     // s_cand is rewritten by the next range
                if (tid == 0) {
                    const unsigned long long at = cn != ~0ull ? cn : (cp != ~0ull ? cp : cm);
                    wc_call c;
                    c.sample = b; c.chrom = slot; c.x = (int)(at >> 32); c.y = (int)(at & 0xffffffffu);
                    c.z = cn != ~0ull ? __longlong_as_double(0x7ff8000000000000ll) : (cp != ~0ull ? INFINITY : -INFINITY);
                    const int slot_i = atomicAdd(&a.ncalls[b], 1);
                    if (slot_i < a.max_calls) a.calls[(size_t)b * a.max_calls + slot_i] = c; else atomicOr(a.status, 1);
                    int spn = s_sp;
                    if ((c.y - lo) + 1 < m - a.min_search) spn = push(spn, c.y + 1, hi);     // triarray.py:79
                    if (c.x - lo > a.min_search) spn = push(spn, lo, c.x);                  // triarray.py:76
                    s_sp = spn;
                }
                continue;
            }
        }
        if (!MINEFF && has_bad) {
            // Run values that contain a NaN, or both +inf and -inf, are NaN; a run with only +inf (-inf) bins is +inf
            // (-inf).  numpy's argmax/argmin return the first NaN entry if there is one (triarray.py:62-66), and a run
            // [x..y] that is NaN makes [lo..y] NaN too, so the first NaN entry is (lo, first y at which [lo..y] turns NaN).
            // Without NaN entries the first +inf entry is the maximum; with only -inf present abs(min) > max picks the
            // first -inf entry (triarray.py:68-70).  Every such value passes `abs(champVal) < threshold` as False.
            if (tid < 3) s_first[tid] = 0x7fffffff;
            __syncthreads();
            for (int i = lo + tid; i < hi; i += SEG_THREADS) {
                const double v = zc[i];
                if (!isfinite(v)) atomicMin(&s_first[isnan(v) ? 0 : (v > 0.0 ? 1 : 2)], i);
            }
            __syncthreads();
            const int fnan = s_first[0], fpos = s_first[1], fneg = s_first[2];
            if (fnan < hi || fpos < hi || fneg < hi) {
                __syncthreads();                     // s_first is rewritten by the next range
                if (tid == 0) {
                    const int both = (fpos < hi && fneg < hi) ? max(fpos, fneg) : 0x7fffffff;
                    const int ynan = min(fnan, both);
                    wc_call c;
                    c.sample = b; c.chrom = slot; c.x = lo;
                    if (ynan < hi) { c.y = ynan; c.z = __longlong_as_double(0x7ff8000000000000ll); }
                    else if (fpos < hi) { c.y = fpos; c.z = INFINITY; }
                    else { c.y = fneg; c.z = -INFINITY; }
                    const int slot_i = atomicAdd(&a.ncalls[b], 1);
                    if (slot_i < a.max_calls) a.calls[(size_t)b * a.max_calls + slot_i] = c; else atomicOr(a.status, 1);
                    if ((c.y - lo) + 1 < m - a.min_search) s_sp = push(s_sp, c.y + 1, hi);   // triarray.py:79 (x == lo: no left part)
                }
                continue;
            }
        }

        // -- sweep by diagonals, in fp32 (it only locates): lane owns the run lengths L0 .. L0+4 (their 1/sqrt in
        //    registers) and walks the start x; P[x] is one broadcast read per step, P[x+L0+r] a 5-deep register window
        //    fed by one conflict-free read.  Per run: FADD, FMNMX(|.|); one FMUL per length at the end --
        float best = 0.f;                             // max over this thread's runs of |score|
        const int ntiles = (m + SEG_TILE - 1) / SEG_TILE;
        {
            for (int round = 0; round * SEG_WARPS < ntiles; ++round) {
                const int t = round * SEG_WARPS + ((round & 1) ? SEG_WARPS - 1 - warp : warp);   // boustrophedon: balance
                if (t >= ntiles) continue;
                const int L0 = 1 + t * SEG_TILE + lane * SEG_R;
                float isq[SEG_R], bh[SEG_R];
#pragma unroll
                for (int r = 0; r < SEG_R; ++r) { isq[r] = (float)__ddiv_rn(1.0, sqrt((double)(L0 + r))); bh[r] = 0.f; }
                int x = lo;
                if (L0 + SEG_R - 1 <= m) {
                    const int xfull = hi - (L0 + SEG_R - 1);       // starts x <= xfull have all five lengths inside [lo, hi)
                    const float* Pq = P + L0;                      // Pq[x + r] = P[x + L0 + r]
                    float ww[SEG_R];                                // slot (j + r) % 5 holds Pq[x + j + r]
#pragma unroll
                    for (int r = 0; r < SEG_R - 1; ++r) ww[r] = Pq[x + r];
                    for (; x + SEG_R - 1 <= xfull; x += SEG_R) {
#pragma unroll
                        for (int j = 0; j < SEG_R; ++j) {
                            ww[(j + SEG_R - 1) % SEG_R] = Pq[x + j + SEG_R - 1];
                            const float px = P[x + j];
#pragma unroll
                            for (int r = 0; r < SEG_R; ++r) {
                                // |fl(d * s)| is non-decreasing in |d| for s > 0 (rounding is monotone): the maximum of the
                                // scores is the score of the largest |difference| - the multiply happens once per length
                                const float v = fabsf(__fsub_rn(ww[(j + r) % SEG_R], px));
                                if (!MINEFF) bh[r] = fmaxf(bh[r], v);
                                else if (v > bh[r] && passes(x + j, L0 + r)) bh[r] = v;   // only record attempts pay
                            }
                        }
                    }
                }
#pragma unroll
                for (int r = 0; r < SEG_R; ++r) {                  // ragged end: the remaining starts of each length
                    const int L = L0 + r;
                    for (int xx = x; xx + L <= hi; ++xx) {
                        const float v = fabsf(__fsub_rn(P[xx + L], P[xx]));
                        if (!MINEFF) bh[r] = fmaxf(bh[r], v);
                        else if (v > bh[r] && passes(xx, L)) bh[r] = v;
                    }
                    bh[r] = __fmul_rn(bh[r], isq[r]);               // the length's extreme score
                    if (L <= m) { dh[L] = bh[r]; best = fmaxf(best, bh[r]); }
                }
            }
        }
        // -- block-wide extreme --
        float bigf = best;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) bigf = fmaxf(bigf, __shfl_xor_sync(0xffffffffu, bigf, o));
        if (lane == 0) s_scan[warp] = __float_as_int(bigf);
        if (tid == 0) s_nrows = 0;
        __syncthreads();
#pragma unroll
        for (int w = 0; w < SEG_WARPS; ++w) bigf = fmaxf(bigf, __int_as_float(s_scan[w]));
        // every run within delta of the true maximum M has an fp32 score >= vlow
        const double big = (double)bigf;
        const double delta = delta_A + 4.0 * 1.1920929e-07 * big;
        if (big + delta < thr_s) continue;            // abs(champVal) < threshold for certain (triarray.py:72-73)
        const float vlow = (float)(big - 2.0 * delta);                  // window floor on the fp32 |score|

        // -- diagonals that can hold the exact champion: those whose own extreme reaches the window --
        for (int L = 1 + tid; L <= m; L += SEG_THREADS) {
            if (dh[L] >= vlow) {
                const int pos = atomicAdd(&s_nrows, 1);
                if (pos < SEG_ROWCAP) s_rows[pos] = L;
            }
        }
        __syncthreads();
        const int nrows_raw = s_nrows;
        const bool all_rows = nrows_raw > SEG_ROWCAP;
        const int nrows = all_rows ? m : nrows_raw;

        // -- exact re-score (numpy order) of every windowed run on those diagonals --
        Best cmax = {-INFINITY, 0x7fffffff, 0x7fffffff}, cmin = {INFINITY, 0x7fffffff, 0x7fffffff};
        for (int ri = 0; ri < nrows; ++ri) {
            const int L = all_rows ? ri + 1 : s_rows[ri];
            const double sq = sqrt((double)L);
            const float isqL = (float)__ddiv_rn(1.0, sq);
            for (int x = lo + tid; x + L <= hi; x += SEG_THREADS) {
                const float av = fabsf(__fmul_rn(__fsub_rn(P[x + L], P[x]), isqL));
                if (av >= vlow && passes(x, L)) {
                    const double sum = np_sum_thread([&](int i) { return zc[x + i]; }, L);     // np_sum(region[x:y+1])
                    Best e = {__ddiv_rn(sum, sq), x, x + L - 1};                                 // / np_sqrt(y-x+1)
                    if (better_max(e, cmax)) cmax = e;
                    if (better_min(e, cmin)) cmin = e;
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const Best om = shfl_best(cmax, o), on = shfl_best(cmin, o);
            if (better_max(om, cmax)) cmax = om;
            if (better_min(on, cmin)) cmin = on;
        }
        if (lane == 0) { s_best[0][warp] = cmax; s_best[1][warp] = cmin; }
        __syncthreads();
        if (tid == 0) {
            for (int w = 0; w < SEG_WARPS; ++w) {
                if (better_max(s_best[0][w], cmax)) cmax = s_best[0][w];
                if (better_min(s_best[1][w], cmin)) cmin = s_best[1][w];
            }
            Best champ = cmax;                                          // triarray.py:62-70
            if (fabs(cmin.v) > champ.v) champ = cmin;
            // Nothing in the window: with the effect-size filter every run of the range is zeroed (0 < threshold, no
            // call); without it the window always holds the sweep's own maximum, so an empty one is an internal error.
            // Either way no champion with x = 0x7fffffff is ever published.
            const bool empty = cmax.x == 0x7fffffff;
            if (empty && !MINEFF) atomicOr(a.status, 8);
            if (!empty && !(fabs(champ.v) < a.thr)) {                   // triarray.py:72-73
                const int slot_i = atomicAdd(&a.ncalls[b], 1);
                if (slot_i < a.max_calls) {
                    wc_call c;
                    c.sample = b; c.chrom = slot; c.x = champ.x; c.y = champ.y; c.z = champ.v;
                    a.calls[(size_t)b * a.max_calls + slot_i] = c;
                } else {
                    atomicOr(a.status, 1);
                }
                int spn = s_sp;
                const int xr = champ.x - lo, yr = champ.y - lo;        // coordinates inside the sub-triangle
                if (yr + 1 < m - a.min_search) spn = push(spn, champ.y + 1, hi);     // triarray.py:79
                if (xr > a.min_search) spn = push(spn, lo, champ.x);                 // triarray.py:76
                s_sp = spn;
            }
        }
    }
}

}  // namespace

extern "C" int wc_segment_batch(wc_ctx* ctx, const double* z_d, const double* r_d, const int32_t* refsizes_d, int N, int B,
                                const int* chrom_bins_h, int nchrom, const int* chromosomes_h, int nsel, int minrefbins,
                                double z_threshold, double mineffectsize, int min_search, double* cwz_d,
                                int32_t* cleaned_bins_d, wc_call* calls_d, int32_t* ncalls_d, int max_calls,
                                void* stream_v) {
    WC_CHECK_ARG(ctx != nullptr && z_d != nullptr && refsizes_d != nullptr && chrom_bins_h != nullptr);
    WC_CHECK_ARG(chromosomes_h != nullptr && cwz_d != nullptr && cleaned_bins_d != nullptr);
    WC_CHECK_ARG(calls_d != nullptr && ncalls_d != nullptr && max_calls > 0);
    WC_CHECK_ARG(N > 0 && B > 0 && nchrom > 0 && nsel > 0 && min_search >= 0);
    // fillTriMin (wisetools.py:475-487): threshold 0 is the plain triangle; a negative threshold keeps every run too
    const bool mineff = mineffectsize > 0.0;
    if (mineff) {
        WC_CHECK_ARG(r_d != nullptr);
        if (!(z_threshold > 0.0)) {
            wc_set_error("segmentation with mineffectsize needs a positive z threshold (zeroed runs would be called)");
            return WC_ERR_ARG;
        }
    }
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    WC_CUDA(cudaSetDevice(ctx->device));
    // abs(m - 1) >= t  <=>  m >= c_hi or m <= c_lo, with c_hi / c_lo the exact double boundaries of the rounded test
    double c_hi = INFINITY, c_lo = -INFINITY;
    if (mineff) {
        const double t = mineffectsize;
        c_hi = 1.0 + t;
        while (c_hi - 1.0 >= t) c_hi = nextafter(c_hi, -INFINITY);
        while (!(c_hi - 1.0 >= t)) c_hi = nextafter(c_hi, INFINITY);
        c_lo = 1.0 - t;
        while (1.0 - c_lo >= t) c_lo = nextafter(c_lo, INFINITY);
        while (!(1.0 - c_lo >= t)) c_lo = nextafter(c_lo, -INFINITY);
    }
    std::vector<int> start(nchrom);
    long long tot = 0;
    for (int c = 0; c < nchrom; ++c) { WC_CHECK_ARG(chrom_bins_h[c] >= 0); start[c] = (int)tot; tot += chrom_bins_h[c]; }
    WC_CHECK_ARG(tot == N);
    // selected chromosomes, longest first (they are the longest-running CTAs)
    std::vector<int> order(nsel);
    int maxlen = 1;
    for (int i = 0; i < nsel; ++i) {
        WC_CHECK_ARG(chromosomes_h[i] >= 0 && chromosomes_h[i] < nchrom);
        order[i] = i;
        maxlen = std::max(maxlen, chrom_bins_h[chromosomes_h[i]]);
    }
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) {
        return chrom_bins_h[chromosomes_h[x]] > chrom_bins_h[chromosomes_h[y]];
    });
    std::vector<int> meta(4 * nsel);
    long long soff = 0;                           // global stack entries per sample before each selected chromosome
    for (int i = 0; i < nsel; ++i) {
        const int c = chromosomes_h[order[i]];
        meta[i] = start[c];
        meta[nsel + i] = chrom_bins_h[c];
        meta[2 * nsel + i] = order[i];
        meta[3 * nsel + i] = (int)soff;
        soff += chrom_bins_h[c] / (min_search + 1) + 1;
    }
    double* zc; double* rcomp = nullptr; int* meta_d; int* status_d;
    int rc;
    if ((rc = wc_reserve(ctx, SLOT_S_ZC, (size_t)B * N * sizeof(double), (void**)&zc))) return rc;
    if (mineff && (rc = wc_reserve(ctx, SLOT_S_RC, (size_t)B * N * sizeof(double), (void**)&rcomp))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_S_META, (size_t)4 * nsel * sizeof(int), (void**)&meta_d))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_S_STATUS, 4 * sizeof(int), (void**)&status_d))) return rc;
    const int pcap = (maxlen + 8) & ~1;
    const size_t aux_bytes = (size_t)pcap * (sizeof(unsigned) + (mineff ? 3 * sizeof(int) : 0));
    size_t smem = (size_t)pcap * sizeof(float) + aux_bytes;
    unsigned* aux_g = nullptr;
    if (smem > 220 * 1024) {                      // keep only the prefix sums in shared memory
        smem = (size_t)pcap * sizeof(float);
        if (smem > 220 * 1024) {
            wc_set_error("segmentation: a chromosome of %d bins needs %zu bytes of shared memory (limit 220 KiB)", maxlen, smem);
            return WC_ERR_ARG;
        }
        if ((rc = wc_reserve(ctx, SLOT_S_AUX, (size_t)nsel * B * aux_bytes, (void**)&aux_g))) return rc;
    }
    // pending-range stack: disjoint ranges longer than min_search.  In shared memory (sized for the longest chromosome)
    // when that costs no resident CTA (it is touched once per range), else in a global slice per CTA sized for its own
    // chromosome: B * sum(len / (min_search + 1) + 1) entries in all.
    const int scap = maxlen / (min_search + 1) + 1;
    const size_t stack_bytes = (size_t)scap * 2 * sizeof(int);
    const void* kfn = mineff ? (const void*)wc_segment_kernel<true> : (const void*)wc_segment_kernel<false>;
    int* stack_g = nullptr;
    bool stack_shared = smem + stack_bytes <= 220 * 1024;
    if (stack_shared) {
        int without = 0, with = 0;
        WC_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem + stack_bytes)));
        WC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&without, kfn, SEG_THREADS, smem));
        WC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&with, kfn, SEG_THREADS, smem + stack_bytes));
        stack_shared = with >= without;
    }
    if (stack_shared) smem += stack_bytes;
    else if ((rc = wc_reserve(ctx, SLOT_S_STACK, (size_t)soff * B * 2 * sizeof(int), (void**)&stack_g))) return rc;
    WC_CUDA(cudaEventRecord(ctx->ev[10], stream));
    WC_CUDA(cudaMemcpyAsync(meta_d, meta.data(), meta.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
    WC_CUDA(cudaMemsetAsync(status_d, 0, 4 * sizeof(int), stream));
    WC_CUDA(cudaMemsetAsync(ncalls_d, 0, (size_t)B * sizeof(int), stream));
    SegArgs a;
    a.z = z_d; a.refsz = refsizes_d; a.N = N; a.B = B; a.sel_start = meta_d; a.sel_len = meta_d + nsel;
    a.sel_slot = meta_d + 2 * nsel; a.sel_soff = meta_d + 3 * nsel; a.nsel = nsel; a.minrefbins = minrefbins; a.thr = z_threshold;
    a.min_search = min_search; a.zc = zc; a.r = r_d; a.rc = rcomp; a.c_hi = c_hi; a.c_lo = c_lo; a.cwz = cwz_d; a.cleaned = cleaned_bins_d; a.calls = calls_d;
    a.ncalls = ncalls_d; a.max_calls = max_calls; a.status = status_d; a.pcap = pcap; a.aux_g = aux_g;
    a.stack_g = stack_g;
    WC_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (mineff) wc_segment_kernel<true><<<(unsigned)((size_t)nsel * B), SEG_THREADS, smem, stream>>>(a);
    else wc_segment_kernel<false><<<(unsigned)((size_t)nsel * B), SEG_THREADS, smem, stream>>>(a);
    WC_CUDA(cudaGetLastError());
    WC_CUDA(cudaEventRecord(ctx->ev[11], stream));
    int status = 0;
    WC_CUDA(cudaMemcpyAsync(&status, status_d, sizeof(int), cudaMemcpyDeviceToHost, stream));
    WC_CUDA(cudaStreamSynchronize(stream));       // meta/status host buffers; the call is documented as synchronous
    ctx->timed_mask |= 1u << 5;
    ctx->counter[6] = 1;
    if (status & 2) { wc_set_error("segmentation: pending ranges overflowed the range stack (internal error)"); return WC_ERR_INTERNAL; }
    if (status & 8) { wc_set_error("segmentation: the error window of a range selected no run"); return WC_ERR_INTERNAL; }
    if (status & 4) {
        wc_set_error("segmentation: the sum of |z| over a chromosome is at least 2^1023 (8.99e307); its run sums could "
                     "overflow double precision");
        return WC_ERR_ARG;
    }
    if (status & 1) { wc_set_error("segmentation: more than max_calls=%d calls for one sample", max_calls); return WC_ERR_ARG; }
    return WC_OK;
}
