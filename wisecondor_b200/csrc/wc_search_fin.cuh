// wisecondor_b200 - K6 in split form: select (wc_finalize_kernel<FT, true>) -> streaming exact re-score -> rank.
// Textually included by wc_search.cu inside its anonymous namespace (uses FinArgs, pair_less and the mbarrier helpers).
#pragma once

// ---------------------------------------------------------------------------------------------------------
// K6a  wc_fin_select_kernel: one WARP per target bin picks its shortlist
// ---------------------------------------------------------------------------------------------------------
// Same decision as step 0-1 of wc_finalize_kernel (entries within the filter's error window of the k-th smallest filter
// distance; everything beyond the row's final threshold dropped first), organised for memory-level parallelism: the row's
// entries sit in ~10 separate buffers (one per K5 segment, plus the incoming buffers) that are cold in L2 when K6 starts,
// and the CTA-per-row kernel walked them source after source - two dependent DRAM round trips per source and warp, 0.77 ms
// at 600 x 50 kb for 0.5 GB.  Here a lane reads the counts of a source each (one round trip), a shared prefix table maps a
// flat entry number to (source, offset), and every lane has SEL_U independent entry loads in flight (second round trip).
// The k-th smallest key is found by integer bisection on keys held in registers (as in prune_row), exact up to ties.
// Rows with more than SEL_ECAP live entries or more than SEL_MAXSRC sources (never-pruned rows of small matrices) go to `big_list`
// and are handled by wc_finalize_kernel<FT, true> afterwards.
constexpr int SEL_WARPS = 4;
constexpr int SEL_ECAP = 1024;               // live entries of a row held by its warp: 32 keys per lane (typical: 400-800)
constexpr int SEL_EPL = SEL_ECAP / 32;
constexpr int SEL_U = 4;                     // entry loads in flight per lane
constexpr int SEL_MAXSRC = 255;           // sources of a row: two per K5 piece of its row block, plus the incoming buffers
constexpr size_t SEL_WARP_BYTES = (size_t)SEL_ECAP * 12 + (SEL_MAXSRC + 1) * 4 + 12;      // keys, bins, prefix table
constexpr size_t SEL_WARP_STRIDE = (SEL_WARP_BYTES + 15) / 16 * 16;

__global__ void __launch_bounds__(SEL_WARPS * 32) wc_fin_select_kernel(const FinArgs a, int* __restrict__ big_list,
                                                                       int* __restrict__ big_count, int* __restrict__ stats) {
    extern __shared__ __align__(16) unsigned char sel_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rloc = blockIdx.x * SEL_WARPS + warp;
    const int rows = a.row_end - a.row_begin;
    if (rloc >= rows) return;
    u64* en_k = reinterpret_cast<u64*>(sel_raw + (size_t)warp * SEL_WARP_STRIDE);
    int* en_j = reinterpret_cast<int*>(en_k + SEL_ECAP);
    int* pre = en_j + SEL_ECAP;                                   // [nsrc + 1] exclusive prefix of the sources' counts
    const int row = a.row_begin + rloc;
    const int rb = rloc / BM, rl = rloc % BM;
    const int seg0 = a.rb_seg_first[rb], nseg = a.rb_seg_count[rb];
    const int nsrc = nseg + (a.in_key != nullptr ? a.in_nsrc : 0);
    int* out_i = a.idx_out + (size_t)rloc * a.k;
    double* out_d = a.dist_out + (size_t)rloc * a.k;
    auto to_big = [&]() {
        if (lane == 0) {
            big_list[atomicAdd(big_count, 1)] = rloc;
            a.sl_p[rloc] = -1;                                     // the fallback kernel overwrites it
        }
    };
    if (nsrc > SEL_MAXSRC) { to_big(); return; }
    // ---- counts and flags of all sources: one round trip ----
    int flagged = 0;
    for (int s0 = 0; s0 < nsrc; s0 += 32) {
        const int s = s0 + lane;
        int n = 0;
        if (s < nsrc) {
            if (s < nseg) {
                n = a.seg_cnt[(size_t)(seg0 + s) * BM + rl];
                flagged |= a.seg_flag[(size_t)(seg0 + s) * BM + rl];
            } else {
                n = a.in_cnt[(size_t)(s - nseg) * a.in_src_rows + rloc];
                if (n > a.in_cap) { flagged = 1; n = a.in_cap; }   // more offers than the buffer holds: exact fallback
            }
        }
        int incl = n;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const int base = s0 == 0 ? 0 : pre[s0];
        if (s < nsrc) pre[s + 1] = base + incl;
        if (s0 == 0 && lane == 0) pre[0] = 0;
        __syncwarp();
    }
    if (__any_sync(0xffffffffu, flagged != 0)) {
        if (lane == 0) {
            a.slow_list[atomicAdd(a.slow_count, 1)] = rloc + a.slow_bias;
            a.sl_p[rloc] = -1;
        }
        return;
    }
    const int total_raw = pre[nsrc];
    const u64 tfinal = a.row_thr != nullptr ? __ldcg(a.row_thr + rloc) : ~0ull;
    // ---- entries: SEL_U independent loads per lane and round; those beyond the row's final threshold are dead weight ----
    int kept = 0;
    for (int t0 = 0; t0 < total_raw; t0 += 32 * SEL_U) {
        u64 key[SEL_U];
        int jj[SEL_U];
#pragma unroll
        for (int u = 0; u < SEL_U; ++u) {
            const int t = t0 + u * 32 + lane;
            key[u] = ~0ull;
            jj[u] = 0;
            if (t < total_raw) {
                int lo = 0, hi = nsrc;                              // largest s with pre[s] <= t
                while (hi - lo > 1) {
                    const int m = (lo + hi) >> 1;
                    if (pre[m] <= t) lo = m; else hi = m;
                }
                const int e = t - pre[lo];
                size_t off;
                const u64* kb;
                const int* jb;
                if (lo < nseg) {
                    off = ((size_t)(seg0 + lo) * BM + rl) * a.cap + e;
                    kb = a.cand_key;
                    jb = a.cand_j;
                } else {
                    off = ((size_t)(lo - nseg) * a.in_src_rows + rloc) * a.in_cap + e;
                    kb = a.in_key;
                    jb = a.in_j;
                }
                key[u] = kb[off];
                jj[u] = jb[off];
            }
        }
#pragma unroll
        for (int u = 0; u < SEL_U; ++u) {
            const bool keep = t0 + u * 32 + lane < total_raw && key[u] <= tfinal;
            const unsigned bm = __ballot_sync(0xffffffffu, keep);
            const int pos = kept + __popc(bm & ((1u << lane) - 1u));
            if (keep && pos < SEL_ECAP) {
                en_k[pos] = key[u];
                en_j[pos] = jj[u];
            }
            kept += __popc(bm);
        }
    }
    if (kept > SEL_ECAP) { to_big(); return; }
    if (kept == 0) {
        for (int e = lane; e < a.k; e += 32) { out_i[e] = -1; out_d[e] = 1e10; }
        if (lane == 0) a.sl_p[rloc] = -1;
        return;
    }
    __syncwarp();
    // ---- k-th smallest key (unsigned order == distance order) by bisection on a register copy ----
    u64 d[SEL_EPL];
#pragma unroll
    for (int t = 0; t < SEL_EPL; ++t) d[t] = t * 32 + lane < kept ? en_k[t * 32 + lane] : ~0ull;
    u64 lo = ~0ull, hi = 0ull;
#pragma unroll
    for (int t = 0; t < SEL_EPL; ++t) {
        if (t * 32 + lane < kept) {
            lo = d[t] < lo ? d[t] : lo;
            hi = d[t] > hi ? d[t] : hi;
        }
    }
    lo = warp_min_u64(lo);
    hi = warp_max_u64(hi);
    u64 blo = lo, bhi = hi, cut = hi;            // count(<= cut) >= min(k, kept) throughout
    int c_hi = kept;
    for (int it = 0; it < 70 && c_hi > a.k; ++it) {
        if (bhi - blo < 2) break;                // bracket exhausted (ties at the k-th place): keep the current cut
        const u64 mid = blo + ((bhi - blo) >> 1);
        int c = 0;
#pragma unroll
        for (int t = 0; t < SEL_EPL; ++t) c += d[t] <= mid ? 1 : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (c >= a.k) { bhi = mid; c_hi = c; cut = mid; } else { blo = mid; }
    }
    u64 vstar = 0ull;
#pragma unroll
    for (int t = 0; t < SEL_EPL; ++t)
        if (d[t] <= cut && d[t] > vstar) vstar = d[t];
    vstar = warp_max_u64(vstar);
    const double dv = dist_of_key(vstar);
    // (filter distances <= 0 - rounding noise of duplicates - order backwards as keys: the window then starts at 0, and their
    // keys, sign bit clear, pass any positive window)
    double window = fmax(dv, 0.0) + a.mcoef * (a.norms[row] + fabs(dv)) + madd_of(a);
    if (!(window > 1e-300)) window = 1e-300;
    const u64 wkey = key_of_tau(window);
    // ---- shortlist: entries within the window, in entry order ----
    int p = 0, jmin = 0x7fffffff;
#pragma unroll
    for (int t = 0; t < SEL_EPL; ++t) {
        const bool keep = t * 32 + lane < kept && d[t] <= wkey;
        const unsigned bm = __ballot_sync(0xffffffffu, keep);
        const int pos = p + __popc(bm & ((1u << lane) - 1u));
        if (keep && pos < a.shortcap) {
            const int j = en_j[t * 32 + lane];
            a.sl_j[(size_t)rloc * a.shortcap + pos] = j;
            jmin = min(jmin, j);
        }
        p += __popc(bm);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) jmin = min(jmin, __shfl_xor_sync(0xffffffffu, jmin, o));
    if (lane == 0) {
        if (p > a.shortcap) {                    // tie plateau wider than the shortlist: exact fallback
            a.slow_list[atomicAdd(a.slow_count, 1)] = rloc + a.slow_bias;
            a.sl_p[rloc] = -1;
        } else {
            a.sl_p[rloc] = p;
            // Work items are filed by the smallest shortlisted bin: target bins that share candidates are re-scored close in
            // time, so their candidate rows are still in the L2 (LRU model on the bench matrix: misses 44 % -> 24 %).
            const int bkt = min(jmin >> a.bkt_shift, FIN_BUCKETS - 1);
            a.sl_b[rloc] = bkt;
            atomicAdd(a.bkt_hist + bkt, (p + 31) >> 5);
            if (stats != nullptr) { atomicAdd(stats, kept); atomicAdd(stats + 1, p); atomicMax(stats + 2, kept); }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// K6a'  wc_fin_select_hist_kernel: the same decision without holding the row's entries (option k6_select = 1)
// ---------------------------------------------------------------------------------------------------------
// The warp-per-row select above keeps a row's live entries in shared memory (12 KB per warp: 16 warps per SM) and rows
// with more than 1024 of them go to the CTA-per-row kernel (most rows at 10 kb).  Here the entries are streamed twice
// and never held: pass 1 histograms the live filter distances over 1024 equal buckets of [0, d(final threshold)]; the
// bucket b* holding the k-th smallest gives v* = its upper edge (a bound of the k-th smallest from above); pass 2 re-reads
// the entries (L2-hot), emits those inside the window of v* and histograms the entries of b* 1024 times finer, which
// tightens v* to 2^-20 of the range: the few entries the finer window excludes are squeezed out of the emitted list in
// place.  Any bound from above gives the same final table; the tight one matters because the re-score's cost goes by
// started groups of 32 candidates (r04a, 2000 x 10 kb: 1.6 % more candidates from the one-level bound, 17 % more re-score
// time).  4 KB of shared memory per warp, 64 registers: 32 warps per SM in flight against the cold buffers' latency, and
// no limit on a row's entries.
constexpr int SELH_WARPS = 8;
constexpr int SELH_BINS = 1024;

__global__ void __launch_bounds__(SELH_WARPS * 32, 5) wc_fin_select_hist_kernel(const FinArgs a, int* __restrict__ big_list,
                                                                            int* __restrict__ big_count, int* __restrict__ stats) {
    __shared__ int s_hist[SELH_WARPS][SELH_BINS];
    __shared__ int s_pre[SELH_WARPS][SEL_MAXSRC + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rloc = blockIdx.x * SELH_WARPS + warp;
    const int rows = a.row_end - a.row_begin;
    if (rloc >= rows) return;
    int* hist = s_hist[warp];
    int* pre = s_pre[warp];
    const int row = a.row_begin + rloc;
    const int rb = rloc / BM, rl = rloc % BM;
    const int seg0 = a.rb_seg_first[rb], nseg = a.rb_seg_count[rb];
    const int nsrc = nseg + (a.in_key != nullptr ? a.in_nsrc : 0);
    int* out_i = a.idx_out + (size_t)rloc * a.k;
    double* out_d = a.dist_out + (size_t)rloc * a.k;
    if (nsrc > SEL_MAXSRC) {
        if (lane == 0) { big_list[atomicAdd(big_count, 1)] = rloc; a.sl_p[rloc] = -1; }
        return;
    }
    for (int b = lane; b < SELH_BINS; b += 32) hist[b] = 0;
    int flagged = 0;
    for (int s0 = 0; s0 < nsrc; s0 += 32) {
        const int s = s0 + lane;
        int n = 0;
        if (s < nsrc) {
            if (s < nseg) {
                n = a.seg_cnt[(size_t)(seg0 + s) * BM + rl];
                flagged |= a.seg_flag[(size_t)(seg0 + s) * BM + rl];
            } else {
                n = a.in_cnt[(size_t)(s - nseg) * a.in_src_rows + rloc];
                if (n > a.in_cap) { flagged = 1; n = a.in_cap; }
            }
        }
        int incl = n;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const int base = s0 == 0 ? 0 : pre[s0];
        if (s < nsrc) pre[s + 1] = base + incl;
        if (s0 == 0 && lane == 0) pre[0] = 0;
        __syncwarp();
    }
    if (__any_sync(0xffffffffu, flagged != 0)) {
        if (lane == 0) { a.slow_list[atomicAdd(a.slow_count, 1)] = rloc + a.slow_bias; a.sl_p[rloc] = -1; }
        return;
    }
    const u64 tfinal = a.row_thr != nullptr ? __ldcg(a.row_thr + rloc) : ~0ull;
    // sweep(f): f(key, bin, valid) for every entry of the row, source by source in rounds of 32 entries (lane = entry), SEL_U
    // rounds' loads in flight; the cursor (source, round) is warp-uniform, so f may vote.  (r04e: a flat entry number mapped
    // to its source by a binary search over the prefix table cost half of the kernel's 6 170 instructions per row.)
    auto sweep = [&](auto&& f) {
        int s = 0, e0 = 0, ns = nsrc > 0 ? pre[1] : 0;           // source, first entry of its next round, its entry count
        bool more = true;
        while (more) {
            u64 key[SEL_U];
            int jj[SEL_U];
            bool ok[SEL_U];
#pragma unroll
            for (int u = 0; u < SEL_U; ++u) {
                while (s < nsrc && e0 >= ns) { ++s; e0 = 0; ns = s < nsrc ? pre[s + 1] - pre[s] : 0; }
                key[u] = ~0ull;
                jj[u] = 0;
                ok[u] = false;
                if (s < nsrc) {
                    const int e = e0 + lane;
                    if (e < ns) {
                        ok[u] = true;
                        if (s < nseg) {
                            const size_t off = ((size_t)(seg0 + s) * BM + rl) * a.cap + e;
                            key[u] = a.cand_key[off];
                            jj[u] = a.cand_j[off];
                        } else {
                            const size_t off = ((size_t)(s - nseg) * a.in_src_rows + rloc) * a.in_cap + e;
                            key[u] = a.in_key[off];
                            jj[u] = a.in_j[off];
                        }
                    }
                    e0 += 32;
                } else {
                    more = false;
                }
            }
#pragma unroll
            for (int u = 0; u < SEL_U; ++u) f(key[u], jj[u], ok[u]);
        }
    };
    // ---- pass 1: histogram of the live filter distances ----
    // bucket scale: distances in [d0, dmax] = [0, the row's final threshold].  A row nobody published a threshold for still
    // carries the initial one (1e10 or 3e38, or ~0 without a table): one more pass for the smallest and largest entry
    // that can be below 1e10 (entries from there on - fillers, inf, NaN - rank last and are dropped at the end,
    // wisetools.py:312-314).  The test is on the filter distance, so it takes the filter's margin: an exact distance just
    // below 1e10 may be filtered a few ulps above it.
    double d0 = 0.0, dmax = dist_of_key(tfinal);
    if (!(dmax < 1e10)) {
        const double cut = 1e10 + a.mcoef * (a.norms[row] + 1e10) + madd_of(a);
        double mn = INFINITY, mx = -INFINITY;
        sweep([&](u64 key, int, bool valid) {
            const double d = dist_of_key(key);
            if (valid && key <= tfinal && d <= cut) { mn = fmin(mn, d); mx = fmax(mx, d); }
        });
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        if (mx >= mn) { d0 = mn; dmax = mx; } else { dmax = 0.0; }          // no entry below 1e10: nothing to shortlist
    }
    // (a span below 1e-5 of the values: one bucket - the upper edge d0 + (b + 1) / scale must not drown in d0's rounding)
    const float scale = dmax - d0 > 1e-5 * fabs(dmax) ? (float)SELH_BINS / (float)(dmax - d0) : 0.0f;
    // bucket of a distance: below d0 -> 0; NaN, inf and anything beyond the range -> the last one (they rank last)
    auto bucket = [&](double d) -> int {
        const float x = (float)(d - d0) * scale;
        return x < (float)SELH_BINS ? (x >= 0.0f ? (int)x : 0) : SELH_BINS - 1;
    };
    int kept = 0;
    sweep([&](u64 key, int, bool valid) {
        const bool live = valid && key <= tfinal;
        if (live) atomicAdd(&hist[bucket(dist_of_key(key))], 1);
        kept += __popc(__ballot_sync(0xffffffffu, live));
    });
    if (kept == 0) {
        for (int e = lane; e < a.k; e += 32) { out_i[e] = -1; out_d[e] = 1e10; }
        if (lane == 0) a.sl_p[rloc] = -1;
        return;
    }
    __syncwarp();
    // ---- the bucket holding the k-th smallest; v* = its upper edge ----
    // kth_bucket(kk, below): the bucket of the kk-th smallest counted entry (-1: fewer than kk) and the number of entries in
    // the buckets before it.  Lane l sums buckets [l * PER, (l + 1) * PER) (reads rotated by the lane: conflict-free), a warp
    // scan finds the lane whose range holds the kk-th, its buckets are then scanned one per lane (PER / 32 rounds).
    auto kth_bucket = [&](int kk, int& below) -> int {
        constexpr int PER = SELH_BINS / 32;
        static_assert(PER % 32 == 0, "one bank per lane in the rotated read");
        int sum = 0;
#pragma unroll 8
        for (int t = 0; t < PER; ++t) sum += hist[lane * PER + ((t + lane) & (PER - 1))];
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const unsigned m = __ballot_sync(0xffffffffu, incl >= kk);
        below = 0;
        if (!m) return -1;
        const int lstar = __ffs(m) - 1;
        int base = __shfl_sync(0xffffffffu, incl - sum, lstar);
        for (int r = 0; r < PER / 32; ++r) {
            const int v = hist[lstar * PER + r * 32 + lane];
            int inc2 = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int w = __shfl_up_sync(0xffffffffu, inc2, o);
                if (lane >= o) inc2 += w;
            }
            const unsigned m2 = __ballot_sync(0xffffffffu, base + inc2 >= kk);
            if (m2) {
                const int l2 = __ffs(m2) - 1;
                below = base + __shfl_sync(0xffffffffu, inc2 - v, l2);
                return lstar * PER + r * 32 + l2;
            }
            base += __shfl_sync(0xffffffffu, inc2, 31);
        }
        return -1;                                               // (not reached: the lane's total covers kk)
    };
    int below = 0;
    int bstar = kth_bucket(a.k, below);
    // every live entry of buckets <= bstar has d - d0 < (bstar + 1) / scale up to the float rounding of the bucket index
    // (conversion, multiply: 2^-23) and of the division below (2 ulp): the edge is taken 2^-20 up.  The last bucket, or fewer
    // than k live entries: all of them, i.e. dmax
    const bool refine = bstar >= 0 && bstar < SELH_BINS - 1 && scale > 0.0f;
    double vstar = dmax;
    if (refine) vstar = fmin(dmax, d0 + (double)(__fdividef((float)(bstar + 1), scale) * (1.0f + 8.0f * 1.1920929e-7f)));
    auto window_key = [&](double v) -> u64 {
        double window = fmax(v, 0.0) + a.mcoef * (a.norms[row] + fabs(v)) + madd_of(a);
        if (!(window > 1e-300)) window = 1e-300;
        const u64 wk = key_of_tau(window);
        return wk > tfinal ? tfinal : wk;                        // never beyond the row's final threshold
    };
    const u64 wkey = window_key(vstar);
    // ---- pass 2: the shortlist under v*'s window (bins to sl_j, keys next to them in the re-score's distance slots), and
    // a second histogram that resolves bucket b* 1024 times finer (the re-score's cost goes by started groups of 32
    // candidates: a shortlist a few entries longer than the exact k-th smallest asks for often starts one more) ----
    // (the refinement pays only where it can save a started group: it takes out about as many entries as pass 1 counted in
    // the bucket of the window's edge - twice that, plus two, is the test after pass 2)
    const int edge_cnt = refine ? hist[bucket(dist_of_key(wkey))] : 0;
    __syncwarp();
    for (int bb = lane; bb < SELH_BINS; bb += 32) hist[bb] = 0;
    __syncwarp();
    const double dscale = (double)scale;
    u64* my_k = a.sl_k + (size_t)rloc * a.shortcap;
    int* my_j = a.sl_j + (size_t)rloc * a.shortcap;
    int p = 0, jmin = 0x7fffffff;
    sweep([&](u64 key, int j, bool valid) {
        const bool keep = valid && key <= wkey;
        const unsigned bm = __ballot_sync(0xffffffffu, keep);
        const int pos = p + __popc(bm & ((1u << lane) - 1u));
        if (keep && pos < a.shortcap) {
            my_j[pos] = j;
            my_k[pos] = key;
            jmin = min(jmin, j);
        }
        p += __popc(bm);
        if (refine && keep) {                                    // (every entry of bucket b* is inside v*'s window)
            const double d = dist_of_key(key);
            if (bucket(d) == bstar) {
                const double f = ((d - d0) * dscale - (double)bstar) * (double)SELH_BINS;
                atomicAdd(&hist[f < (double)SELH_BINS ? (f >= 0.0 ? (int)f : 0) : SELH_BINS - 1], 1);
            }
        }
    });
    if (p > a.shortcap) {                                        // tie plateau wider than the shortlist: exact fallback
        if (lane == 0) {
            a.slow_list[atomicAdd(a.slow_count, 1)] = rloc + a.slow_bias;
            a.sl_p[rloc] = -1;
        }
        return;
    }
    __syncwarp();
    if (refine && p > a.k && ((p - 1) >> 5) != ((max(a.k, p - 2 * edge_cnt - 2) - 1) >> 5)) {
        int below2 = 0;
        const int sstar = kth_bucket(a.k - below, below2);
        // sub-bucket s of b* holds (d - d0) * scale in [b* + s / 1024, b* + (s + 1) / 1024) (the ends of b* clamp into the
        // first and the last one): below the last one its upper edge, a thousandth of its width up for the rounding of
        // f, bounds the k-th smallest
        if (sstar >= 0 && sstar < SELH_BINS - 1) {
            const double v2 = d0 + ((double)bstar + ((double)(sstar + 1) + 1e-3) / (double)SELH_BINS) / dscale;
            const u64 wkey2 = window_key(fmin(vstar, v2));
            if (wkey2 < wkey) {                                  // drop what the finer bound excludes, order kept
                int q = 0;
                jmin = 0x7fffffff;
                for (int e0 = 0; e0 < p; e0 += 32) {
                    const int e = e0 + lane;
                    const bool keep = e < p && __ldcg(my_k + e) <= wkey2;
                    const int j = e < p ? __ldcg(my_j + e) : 0;
                    __syncwarp();                                // slots of this round are read before any is rewritten
                    const unsigned bm = __ballot_sync(0xffffffffu, keep);
                    if (keep) {
                        my_j[q + __popc(bm & ((1u << lane) - 1u))] = j;
                        jmin = min(jmin, j);
                    }
                    q += __popc(bm);
                }
                p = q;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) jmin = min(jmin, __shfl_xor_sync(0xffffffffu, jmin, o));
    if (lane == 0) {
        a.sl_p[rloc] = p;
        const int bkt = min(jmin >> a.bkt_shift, FIN_BUCKETS - 1);
        a.sl_b[rloc] = bkt;
        atomicAdd(a.bkt_hist + bkt, (p + 31) >> 5);
        if (stats != nullptr) { atomicAdd(stats, kept); atomicAdd(stats + 1, p); atomicMax(stats + 2, kept); }
    }
}

// The re-score's work list in locality order: exclusive scan of the buckets' item counts (one CTA), then every row files its
// items under its bucket (order inside a bucket: arrival).
__global__ void __launch_bounds__(FIN_BUCKETS) wc_fin_bucket_scan_kernel(int* __restrict__ hist, int* __restrict__ total) {
    __shared__ int s_w[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int v = hist[tid];
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    int base = 0;
    for (int w = 0; w < warp; ++w) base += s_w[w];
    hist[tid] = base + incl - v;                               // becomes the bucket's cursor
    if (tid == FIN_BUCKETS - 1) *total = base + incl;
}

__global__ void wc_fin_bucket_scatter_kernel(int rows, const int* __restrict__ sl_p, const int* __restrict__ sl_b,
                                             int* __restrict__ cursor, int* __restrict__ grp) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const int p = sl_p[r];
    if (p <= 0) return;
    const int ng = (p + 31) >> 5;
    const int base = atomicAdd(cursor + sl_b[r], ng);
    for (int g = 0; g < ng; ++g) grp[base + g] = (r << 4) | g;
}

// ---------------------------------------------------------------------------------------------------------
// K6c  wc_fin_rescore_kernel<W, NP>: the exact distances of every shortlisted (target bin, candidate bin) pair
// ---------------------------------------------------------------------------------------------------------
// getRefForBins' distance (/root/reference/wisetools.py:302 on Fortran-ordered operands): sum over the samples, strictly in
// sample order, of separately rounded (x_j - x_i)^2.  The arithmetic is a 3-instruction dependent chain per sample and per
// candidate - nothing to speed up there; what bounds the step is bringing ~125 candidate rows of S doubles per target bin
// (28 GB at 600 x 50 kb, 466 GB at 2000 x 10 kb) to the threads.  Register-streaming loads (the fused kernel: one 32-byte
// sector per lane and instruction, 32 different lines per warp instruction) hold the L1 tag stage at one line per cycle:
// ~60 % of its throughput is all the kernel got, at 53 % of L2 and 30 % of DRAM throughput.  Here the rows never pass through L1:
//   * one persistent CTA per SM, W consumer warps + NP producer warps, a ring of NSLOT shared-memory slots;
//   * a work item = 32 shortlist slots of one target bin; a slot holds one chunk (C samples) of the 32 candidate rows and of
//     the target's own row, each brought by ONE bulk copy (cp.async.bulk global -> shared, SASS UBLKCP, C * 8 contiguous
//     bytes) that completes on the slot's mbarrier - the producer lanes only issue, nothing is staged through registers;
//   * a consumer lane owns one candidate: it walks its row of the slot with 128-bit shared-memory loads (rows are
//     C * 8 + 16 bytes apart, an odd number of 16-byte units: conflict-free) against the broadcast target chunk;
//   * items are interleaved over CTAs and warps: item G = (wave * W + w) * gridDim + block; every consumer warp has a private
//     ring of D = NSLOT / W slots which its chunks (wave * nchunks + c) walk round-robin - one producer and one consumer per
//     slot, both in order, so a phase parity names a use unambiguously.
struct RescoreArgs {
    const double* X;
    int S;
    int row_begin;
    int shortcap;
    const int* sl_j;
    double* sl_d;            // [rows][shortcap] exact distances, slot for slot
    const int* sl_p;
    const int* grp;
    const int* grp_count;
    int C;                   // samples per chunk (multiple of 4)
    int nchunks;
    int stride;              // bytes between two rows of a slot: C * 8 + 16 (gather4: box width * 8, rows of a group contiguous)
    int nslot;               // W * D ring slots
    // gather4 form: a slot = 8 groups of 4 rows (one TMA request each) G bytes apart, then the target's chunk
    int gstride;             // G: bytes between two groups (a multiple of 128)
    int slot_bytes;
};

constexpr int RS_HEADER = 1024;       // mbarriers: full[64], empty[64]
constexpr int RS_MAX_SLOTS = 64;

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// One TMA request for FOUR candidate rows: tile::gather4 of a 2-D tensor map over X with a (box width x 1 row) box.
__device__ __forceinline__ void tma_gather4(uint32_t dst, const CUtensorMap* map, int col, int r0, int r1, int r2, int r3, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(col), "r"(r0), "r"(r1), "r"(r2), "r"(r3), "r"(smem_u32(bar))
        : "memory");
}
constexpr int RS_G4_SHIFT = 8;        // odd groups start 8 samples early: their rows sit 64 bytes further -> conflict-free 128-bit loads

// G4 (option k6_g4, off by default): the candidate rows arrive four per TMA request (tile::gather4) instead of one bulk copy
// each - 9 requests per slot instead of 33 (profiles/l2_peak_r03u.json: 24 requests / us / SM from one issuing warp for 1, 2
// or 3.2 KB per request).  Measured r03v: 2.81 against 2.71 ms - the request rate is not what bounds the kernel, the
// shared-memory bandwidth is (every operand byte is written once by the TMA unit and read once by a lane).  The four rows
// of a group land contiguously (box width * 8 bytes apart, an odd number of 16-byte units), the groups G bytes apart (TMA
// destinations are 128-byte aligned); odd groups read their box RS_G4_SHIFT samples early, so that the eight lanes of a
// 128-bit shared-memory load phase (two groups) touch eight different bank groups.
template <int W, int R, bool G4>      // W consumer warps, R producer warps per consumer warp
__global__ void __launch_bounds__((W + W * R) * 32, 1) wc_fin_rescore_kernel(const __grid_constant__ CUtensorMap xmap, const RescoreArgs a) {
    extern __shared__ __align__(128) unsigned char rs_raw[];
    uint64_t* full = reinterpret_cast<uint64_t*>(rs_raw);
    uint64_t* empty = full + RS_MAX_SLOTS;
    const uint32_t slots_u32 = smem_u32(rs_raw + RS_HEADER);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nslot = a.nslot;
    const int D = nslot / W;                   // ring depth per consumer warp
    const uint32_t slot_bytes = G4 ? (uint32_t)a.slot_bytes : 33u * (uint32_t)a.stride;
    if (tid == 0) {
        for (int s = 0; s < nslot; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 32); }      // every consumer lane releases its slot itself
        mbar_fence_init();
        if (G4) tma_prefetch_desc(&xmap);
    }
    __syncthreads();
    const int ngroups = *a.grp_count;
    const int grid = gridDim.x, b = blockIdx.x;
    const int per_wave = W * grid;
    const int nfull = ngroups / per_wave;
    const int rem = ngroups - nfull * per_wave;
    const int nact = rem > b ? (rem - b + grid - 1) / grid : 0;      // warps of this CTA with an item in the last wave
    const int nwaves = nfull + (nact > 0 ? 1 : 0);
    const int nchunks = a.nchunks, C = a.C;
    const size_t row_bytes = (size_t)a.S * 8;

    if (warp < W) {
        // ===== consumers: lane = candidate =====
        const int w = warp;
        for (int wave = 0; wave < nwaves; ++wave) {
            const int wact = wave < nfull ? W : nact;
            if (w >= wact) break;
            const int desc = a.grp[(size_t)(wave * W + w) * grid + b];
            const int rloc = desc >> 4, gi = desc & 15;
            const int p = a.sl_p[rloc];
            const int cnt = min(32, p - gi * 32);
            const int mylane = lane < cnt ? lane : cnt - 1;          // idle lanes shadow the last candidate
            double acc = 0.0;
            const int k0 = wave * nchunks;
            for (int c = 0; c < nchunks; ++c) {
                const int use = (k0 + c) / D, slot = w * D + (k0 + c) - use * D;
                mbar_wait(&full[slot], (uint32_t)(use & 1));
                const uint32_t sb = slots_u32 + (uint32_t)slot * slot_bytes;
                // gather4: every lane has a row of its own (idle lanes: a duplicate of the last candidate's)
                const uint32_t cb = G4 ? sb + (uint32_t)(lane >> 2) * (uint32_t)a.gstride + (uint32_t)(lane & 3) * (uint32_t)a.stride +
                                             (((lane >> 2) & 1) ? RS_G4_SHIFT * 8u : 0u)
                                       : sb + (uint32_t)mylane * (uint32_t)a.stride;
                const uint32_t xb = G4 ? sb + 8u * (uint32_t)a.gstride : sb + 32u * (uint32_t)a.stride;
                const int n = min(C, a.S - c * C);                   // even
                int t = 0;
                for (; t + 8 <= n; t += 8) {
                    double v[8], x[8];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        lds_v2f64(cb + (uint32_t)(t + 2 * u) * 8u, v[2 * u], v[2 * u + 1]);
                        lds_v2f64(xb + (uint32_t)(t + 2 * u) * 8u, x[2 * u], x[2 * u + 1]);
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const double d = __dsub_rn(v[u], x[u]);
                        acc = __dadd_rn(acc, __dmul_rn(d, d));
                    }
                }
                for (; t < n; t += 2) {
                    double v0, v1, x0, x1;
                    lds_v2f64(cb + (uint32_t)t * 8u, v0, v1);
                    lds_v2f64(xb + (uint32_t)t * 8u, x0, x1);
                    double d = __dsub_rn(v0, x0);
                    acc = __dadd_rn(acc, __dmul_rn(d, d));
                    d = __dsub_rn(v1, x1);
                    acc = __dadd_rn(acc, __dmul_rn(d, d));
                }
                mbar_arrive(&empty[slot]);       // (release: this lane's reads of the slot are done)
            }
            if (lane < cnt) a.sl_d[(size_t)rloc * a.shortcap + gi * 32 + lane] = acc;
        }
    } else {
        // ===== producers: warp (w, r) issues the copies of the lanes l = r (mod R) of consumer warp w's slots =====
        // A per-lane bulk copy is a serial loop over the active lanes (UBLKCP takes uniform operands: ~70 cycles per copy and
        // warp, measured) - the issue rate, not the memory system, bounds the kernel unless several warps share a slot's copies.
        const int w = (warp - W) % W, r = (warp - W) / W;
        const bool mine = lane % R == r;
        for (int wave = 0; wave < nwaves; ++wave) {
            const int wact = wave < nfull ? W : nact;
            if (w >= wact) break;
            const int desc = a.grp[(size_t)(wave * W + w) * grid + b];
            const int rloc = desc >> 4, gi = desc & 15;
            const int p = a.sl_p[rloc];
            const int cnt = min(32, p - gi * 32);
            const double* src = nullptr;
            if (!G4 && mine && lane < cnt) src = a.X + (size_t)a.sl_j[(size_t)rloc * a.shortcap + gi * 32 + lane] * a.S;
            int j0 = 0, j1 = 0, j2 = 0, j3 = 0;
            bool issue = false;
            if (G4) {      // lane 4q holds the four bins of group q (lanes beyond the item's candidates repeat its last one)
                j0 = a.sl_j[(size_t)rloc * a.shortcap + gi * 32 + min(lane, cnt - 1)];
                j1 = __shfl_down_sync(0xffffffffu, j0, 1);
                j2 = __shfl_down_sync(0xffffffffu, j0, 2);
                j3 = __shfl_down_sync(0xffffffffu, j0, 3);
                issue = (lane & 3) == 0 && (lane >> 2) % R == r;
            }
            const double* xsrc = a.X + (size_t)(a.row_begin + rloc) * a.S;
            const int k0 = wave * nchunks;
            for (int c = 0; c < nchunks; ++c) {
                const uint32_t bytes = (uint32_t)min(C, a.S - c * C) * 8u;
                const size_t off = (size_t)c * C;
                const int use = (k0 + c) / D, slot = w * D + (k0 + c) - use * D;
                if (use > 0) mbar_wait(&empty[slot], (uint32_t)((use - 1) & 1));
                const uint32_t sb = slots_u32 + (uint32_t)slot * slot_bytes;
                if (G4) {
                    if (r == 0 && lane == 0) {      // a box counts in full, also where it reaches beyond the row (zero fill)
                        mbar_arrive_expect_tx(&full[slot], 32u * (uint32_t)a.stride + bytes);
                        bulk_g2s(sb + 8u * (uint32_t)a.gstride, xsrc + off, bytes, &full[slot]);
                    }
                    if (issue) {
                        const int q = lane >> 2;
                        tma_gather4(sb + (uint32_t)q * (uint32_t)a.gstride, &xmap, c * C - ((q & 1) ? RS_G4_SHIFT : 0), j0, j1, j2, j3, &full[slot]);
                    }
                } else {
                    if (r == 0 && lane == 0) {
                        mbar_arrive_expect_tx(&full[slot], (uint32_t)(cnt + 1) * bytes);
                        bulk_g2s(sb + 32u * (uint32_t)a.stride, xsrc + off, bytes, &full[slot]);
                    }
                    if (src != nullptr) bulk_g2s(sb + (uint32_t)lane * (uint32_t)a.stride, src + off, bytes, &full[slot]);
                }
            }
        }
    }
    (void)row_bytes;
}

// ---------------------------------------------------------------------------------------------------------
// K6d  wc_fin_rank_kernel: one warp per target bin ranks its re-scored shortlist by (distance, bin) and writes the first k
// ---------------------------------------------------------------------------------------------------------
struct RankArgs {
    int rows, k, shortcap;
    const int* sl_j;
    const double* sl_d;
    const int* sl_p;
    const int* row_cs;
    const int* row_ce;
    int row_begin;
    int* idx_out;
    double* dist_out;
};
constexpr int RK_WARPS = 8;

// (key a, bin ja) < (key b, bin jb) as one 96-bit subtraction with borrow: 0xffffffff if less, else 0
__device__ __forceinline__ unsigned pair_less96(u64 a, int ja, u64 b, int jb) {
    unsigned r;
    asm("{\n"
        ".reg .u32 t;\n"
        "sub.cc.u32 t, %1, %4;\n"
        "subc.cc.u32 t, %2, %5;\n"
        "subc.cc.u32 t, %3, %6;\n"
        "subc.u32 %0, 0, 0;\n"
        "}\n"
        : "=r"(r)
        : "r"((unsigned)ja), "r"((unsigned)(a & 0xffffffffu)), "r"((unsigned)(a >> 32)), "r"((unsigned)jb),
          "r"((unsigned)(b & 0xffffffffu)), "r"((unsigned)(b >> 32)));
    return r;
}

// One compare-exchange step at distance STRIDE of the bitonic network (blocks of `size` sort up / down alternately).
// Pairs are distinct except for padding entries, which are identical - either choice is the same.
template <int EPL, int STRIDE>
__device__ __forceinline__ void rank_step(u64 (&key)[EPL], int (&bin)[EPL], int lane, int size) {
#pragma unroll
    for (int t = 0; t < EPL; ++t) {
        const int e = t * 32 + lane;
        const bool up = (e & size) == 0;                    // this block sorts ascending
        if (STRIDE >= 32) {
            const int t2 = t ^ (STRIDE >> 5);
            if (t2 > t) {                                    // one compare-exchange per pair, both ends in this lane
                const bool less2 = pair_less96(key[t2], bin[t2], key[t], bin[t]) != 0u;
                if (less2 == up) {
                    const u64 tk = key[t]; key[t] = key[t2]; key[t2] = tk;
                    const int tb = bin[t]; bin[t] = bin[t2]; bin[t2] = tb;
                }
            }
        } else {
            const u64 ok = __shfl_xor_sync(0xffffffffu, key[t], STRIDE);
            const int ob = __shfl_xor_sync(0xffffffffu, bin[t], STRIDE);
            const bool want_min = ((lane & STRIDE) == 0) == up;       // this end keeps the smaller one
            const bool other_less = pair_less96(ok, ob, key[t], bin[t]) != 0u;
            if (other_less == want_min) { key[t] = ok; bin[t] = ob; }
        }
    }
}

// Bitonic sort of 32 * EPL (key, bin) pairs held EPL per lane (element e = t * 32 + lane), ascending by (key, bin):
// compare-exchange distances below 32 go through shuffles, the others stay inside the lane.  The loop over the block size is
// a run-time loop around ONE copy of every distance's step (the fully unrolled network is 0.7 MB of code for the three
// instantiations).
template <int EPL>
__device__ __forceinline__ void rank_sort(u64 (&key)[EPL], int (&bin)[EPL], int lane) {
#pragma unroll 1
    for (int size = 2; size <= 32 * EPL; size <<= 1) {
        if (EPL >= 16 && size > 256) rank_step<EPL, (EPL >= 16 ? 256 : 1)>(key, bin, lane, size);
        if (EPL >= 8 && size > 128) rank_step<EPL, (EPL >= 8 ? 128 : 1)>(key, bin, lane, size);
        if (EPL >= 4 && size > 64) rank_step<EPL, (EPL >= 4 ? 64 : 1)>(key, bin, lane, size);
        if (EPL >= 2 && size > 32) rank_step<EPL, (EPL >= 2 ? 32 : 1)>(key, bin, lane, size);
        if (size > 16) rank_step<EPL, 16>(key, bin, lane, size);
        if (size > 8) rank_step<EPL, 8>(key, bin, lane, size);
        if (size > 4) rank_step<EPL, 4>(key, bin, lane, size);
        if (size > 2) rank_step<EPL, 2>(key, bin, lane, size);
        rank_step<EPL, 1>(key, bin, lane, size);
    }
}

template <int EPL>
__device__ __forceinline__ void rank_row(const RankArgs& a, int rloc, int p, int lane) {
    u64 key[EPL];
    int bin[EPL];
    int nvalid = 0;
#pragma unroll
    for (int t = 0; t < EPL; ++t) {
        const int e = t * 32 + lane;
        key[t] = ~0ull;                                              // padding sorts last
        bin[t] = 0x7fffffff;
        if (e < p) {
            const double d = a.sl_d[(size_t)rloc * a.shortcap + e];
            const bool ok = d < 1e10;       // wisetools.py:312-314: strict `<` against the 1e10 start value; NaN fails
            // distances are sums of squares: their bit patterns order like unsigned integers (no FP64 compare in the sort)
            if (ok) { key[t] = (u64)__double_as_longlong(d); bin[t] = a.sl_j[(size_t)rloc * a.shortcap + e]; }
            nvalid += ok ? 1 : 0;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nvalid += __shfl_xor_sync(0xffffffffu, nvalid, o);
    rank_sort<EPL>(key, bin, lane);
    const int row = a.row_begin + rloc;
    const int cs = a.row_cs[row], ce = a.row_ce[row];
    int* out_i = a.idx_out + (size_t)rloc * a.k;
    double* out_d = a.dist_out + (size_t)rloc * a.k;
    const int nout = nvalid < a.k ? nvalid : a.k;
#pragma unroll
    for (int t = 0; t < EPL; ++t) {
        const int e = t * 32 + lane;
        if (e < nout) {
            out_i[e] = bin[t] >= ce ? bin[t] - (ce - cs) : bin[t];
            out_d[e] = __longlong_as_double((long long)key[t]);
        }
    }
    for (int e = nvalid + lane; e < a.k; e += 32) { out_i[e] = -1; out_d[e] = 1e10; }
}

__global__ void __launch_bounds__(RK_WARPS * 32) wc_fin_rank_kernel(const RankArgs a) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rloc = blockIdx.x * RK_WARPS + warp;
    if (rloc >= a.rows) return;
    const int p = a.sl_p[rloc];
    if (p < 0) return;                                          // fillers written by the select, or the exhaustive kernel's row
    if (p <= 128) rank_row<4>(a, rloc, p, lane);
    else if (p <= 256) rank_row<8>(a, rloc, p, lane);
    else rank_row<16>(a, rloc, p, lane);
}

// ---------------------------------------------------------------------------------------------------------
// host: K6 of a search call (both the single-GPU call and the finish of a sharded symmetric search)
// ---------------------------------------------------------------------------------------------------------
template <int W, int R>
static int launch_rescore(const RescoreArgs& ra, const CUtensorMap& xmap, bool g4, int grid, size_t smem, cudaStream_t stream) {
    if (g4) {
        WC_CUDA(cudaFuncSetAttribute(wc_fin_rescore_kernel<W, R, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        wc_fin_rescore_kernel<W, R, true><<<grid, (W + W * R) * 32, smem, stream>>>(xmap, ra);
        return WC_OK;
    }
    WC_CUDA(cudaFuncSetAttribute(wc_fin_rescore_kernel<W, R, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    wc_fin_rescore_kernel<W, R, false><<<grid, (W + W * R) * 32, smem, stream>>>(xmap, ra);
    return WC_OK;
}

// Returns the number of kernel launches through *launches.  fa.sl_* / fa.grp* are filled here.
static int launch_finalize(wc_ctx* ctx, cudaStream_t stream, FinArgs fa, int rows, bool wide, long long* launches) {
    const size_t fin_smem = (size_t)FIN_ECAP * 12 + (size_t)fa.shortcap * 12 + HIST_BINS * 4;
    // the streaming re-score needs 16-byte aligned rows (bulk copies): an even number of samples
    const bool split = ctx->k6_split != 0 && fa.S % 2 == 0 && fa.S >= 8 && (reinterpret_cast<uintptr_t>(fa.X) & 15) == 0 && rows > 0;
    fa.sl_j = nullptr; fa.sl_p = nullptr; fa.grp = nullptr; fa.grp_count = nullptr; fa.row_list = nullptr; fa.row_count = nullptr; fa.stats = nullptr;
    ctx->k6_stats_d = nullptr;
    ctx->phase_ms[10] = 0.0;
    ctx->timed_mask &= ~(1u << 10);
    if (!split) {
        if (wide) {
            WC_CUDA(cudaFuncSetAttribute(wc_finalize_kernel<160, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fin_smem));
            wc_finalize_kernel<160, false><<<rows, 160, fin_smem, stream>>>(fa);
        } else {
            WC_CUDA(cudaFuncSetAttribute(wc_finalize_kernel<FIN_THREADS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fin_smem));
            wc_finalize_kernel<FIN_THREADS, false><<<rows, FIN_THREADS, fin_smem, stream>>>(fa);
        }
        WC_CUDA(cudaGetLastError());
        *launches = 1;
        return WC_OK;
    }
    int rc;
    double* sl_d;
    const int gpr = fa.shortcap / 32;                      // work items per row at most
    if ((rc = wc_reserve(ctx, SLOT_FIN_J, (size_t)rows * fa.shortcap * sizeof(int), (void**)&fa.sl_j))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_FIN_D, (size_t)rows * fa.shortcap * sizeof(double), (void**)&sl_d))) return rc;
    fa.sl_k = reinterpret_cast<u64*>(sl_d);               // K6a' parks the shortlisted keys where K6c later writes the distances
    if ((rc = wc_reserve(ctx, SLOT_FIN_P, (2 * (size_t)rows + 8 + FIN_BUCKETS) * sizeof(int), (void**)&fa.sl_p))) return rc;
    if ((rc = wc_reserve(ctx, SLOT_FIN_GRP, (size_t)rows * (gpr + 1) * sizeof(int), (void**)&fa.grp))) return rc;
    // sl_p[rows .. rows + 3]: work-item counter, rows passed on to the CTA-per-row select, live entries / shortlist sizes (stats)
    fa.grp_count = fa.sl_p + rows;
    int* big_count = fa.sl_p + rows + 1;
    int* stats = fa.sl_p + rows + 2;
    fa.sl_b = fa.sl_p + rows + 8;
    fa.bkt_hist = fa.sl_b + rows;
    fa.bkt_shift = 0;
    while (((fa.N - 1) >> fa.bkt_shift) >= FIN_BUCKETS) ++fa.bkt_shift;
    WC_CUDA(cudaMemsetAsync(fa.bkt_hist, 0, FIN_BUCKETS * sizeof(int), stream));
    int* big_list = fa.grp + (size_t)rows * gpr;
    WC_CUDA(cudaMemsetAsync(fa.grp_count, 0, 5 * sizeof(int), stream));
    fa.row_list = nullptr; fa.row_count = nullptr; fa.stats = stats;
    if (ctx->k6_select != 0) {
        wc_fin_select_hist_kernel<<<(rows + SELH_WARPS - 1) / SELH_WARPS, SELH_WARPS * 32, 0, stream>>>(fa, big_list, big_count, stats);
    } else {
        const size_t sel_smem = SEL_WARPS * SEL_WARP_STRIDE;
        WC_CUDA(cudaFuncSetAttribute(wc_fin_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sel_smem));
        wc_fin_select_kernel<<<(rows + SEL_WARPS - 1) / SEL_WARPS, SEL_WARPS * 32, sel_smem, stream>>>(fa, big_list, big_count, stats);
    }
    WC_CUDA(cudaGetLastError());
    {   // rows with more live entries than a warp holds (never-pruned rows of small matrices): the CTA-per-row select
        fa.row_list = big_list; fa.row_count = big_count;
        const int g = std::min(rows, 8 * ctx->sm_count);
        if (wide) {
            WC_CUDA(cudaFuncSetAttribute(wc_finalize_kernel<160, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fin_smem));
            wc_finalize_kernel<160, true><<<g, 160, fin_smem, stream>>>(fa);
        } else {
            WC_CUDA(cudaFuncSetAttribute(wc_finalize_kernel<FIN_THREADS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fin_smem));
            wc_finalize_kernel<FIN_THREADS, true><<<g, FIN_THREADS, fin_smem, stream>>>(fa);
        }
        WC_CUDA(cudaGetLastError());
    }
    wc_fin_bucket_scan_kernel<<<1, FIN_BUCKETS, 0, stream>>>(fa.bkt_hist, fa.grp_count);
    wc_fin_bucket_scatter_kernel<<<(rows + 255) / 256, 256, 0, stream>>>(rows, fa.sl_p, fa.sl_b, fa.bkt_hist, fa.grp);
    WC_CUDA(cudaGetLastError());
    WC_CUDA(cudaEventRecord(ctx->ev[20], stream));
    RescoreArgs ra;
    ra.X = fa.X; ra.S = fa.S; ra.row_begin = fa.row_begin; ra.shortcap = fa.shortcap; ra.sl_j = fa.sl_j; ra.sl_d = sl_d;
    ra.sl_p = fa.sl_p; ra.grp = fa.grp; ra.grp_count = fa.grp_count;
    const int W = ctx->k6_warps > 0 ? ctx->k6_warps : 4;
    const int R = ctx->k6_prod > 0 ? ctx->k6_prod : 2;
    // gather4 form: four candidate rows per TMA request (needs the tensor-map encoder and a matrix of at least one box)
    bool g4 = ctx->k6_g4 != 0 && ctx->encode_tiled != nullptr && fa.S >= 64 && fa.N >= 4;
    int C = ctx->k6_chunk > 0 ? ctx->k6_chunk : (g4 ? 86 : 100);
    CUtensorMap xmap;
    memset(&xmap, 0, sizeof(xmap));
    size_t slot_bytes = 0;
    if (g4) {
        // chunks of about C samples that tile S evenly; box = chunk + RS_G4_SHIFT samples, half of it an odd number (rows of
        // a group an odd number of 16-byte units apart)
        const int nch = (fa.S + C - 1) / C;
        C = (fa.S + nch - 1) / nch;
        C += C & 1;
        if ((((C + RS_G4_SHIFT) / 2) & 1) == 0) C += 2;
        const int cbox = C + RS_G4_SHIFT;
        if (cbox > 256) g4 = false;
        else {
            ra.C = C;
            ra.nchunks = (fa.S + C - 1) / C;
            ra.stride = cbox * 8;
            ra.gstride = (4 * ra.stride + 127) / 128 * 128;
            ra.slot_bytes = 8 * ra.gstride + (C * 8 + 127) / 128 * 128;
            slot_bytes = (size_t)ra.slot_bytes;
            cuuint64_t dims[2] = {(cuuint64_t)fa.S, (cuuint64_t)fa.N};
            cuuint64_t strides[1] = {(cuuint64_t)fa.S * sizeof(double)};
            cuuint32_t box[2] = {(cuuint32_t)cbox, 1};
            cuuint32_t estr[2] = {1, 1};
            CUresult r = reinterpret_cast<PFN_encodeTiled>(ctx->encode_tiled)(
                &xmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(fa.X), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) g4 = false;
        }
    }
    if (!g4) {
        C = ctx->k6_chunk > 0 ? ctx->k6_chunk : 100;
        C = std::max(4, std::min(C & ~3, 480));
        if (C > fa.S) C = (fa.S + 3) & ~3;
        ra.C = C;
        ra.nchunks = (fa.S + C - 1) / C;
        ra.stride = C * 8 + 16;
        ra.gstride = 0; ra.slot_bytes = 0;
        slot_bytes = (size_t)33 * ra.stride;
    }
    ra.nslot = (int)std::min<size_t>(RS_MAX_SLOTS, ((size_t)226 * 1024 - RS_HEADER) / slot_bytes);
    if (ra.nslot < 2 * W) { wc_set_error("K6: chunk of %d samples leaves %d ring slots for %d consumer warps", C, ra.nslot, W); return WC_ERR_ARG; }
    ra.nslot = ra.nslot / W * W;
    const size_t smem = RS_HEADER + (size_t)ra.nslot * slot_bytes;
    const int grid = ctx->sm_count;
    if (W == 2 && R == 4) rc = launch_rescore<2, 4>(ra, xmap, g4, grid, smem, stream);
    else if (W == 2 && R == 8) rc = launch_rescore<2, 8>(ra, xmap, g4, grid, smem, stream);
    else if (W == 4 && R == 1) rc = launch_rescore<4, 1>(ra, xmap, g4, grid, smem, stream);
    else if (W == 4 && R == 2) rc = launch_rescore<4, 2>(ra, xmap, g4, grid, smem, stream);
    else if (W == 4 && R == 4) rc = launch_rescore<4, 4>(ra, xmap, g4, grid, smem, stream);
    else if (W == 4 && R == 7) rc = launch_rescore<4, 7>(ra, xmap, g4, grid, smem, stream);
    else if (W == 8 && R == 1) rc = launch_rescore<8, 1>(ra, xmap, g4, grid, smem, stream);
    else if (W == 8 && R == 2) rc = launch_rescore<8, 2>(ra, xmap, g4, grid, smem, stream);
    else if (W == 8 && R == 3) rc = launch_rescore<8, 3>(ra, xmap, g4, grid, smem, stream);
    else { wc_set_error("K6: no kernel for %d consumer warps x %d producer warps each", W, R); return WC_ERR_ARG; }
    if (rc) return rc;
    WC_CUDA(cudaGetLastError());
    WC_CUDA(cudaEventRecord(ctx->ev[21], stream));
    RankArgs ka;
    ka.rows = rows; ka.k = fa.k; ka.shortcap = fa.shortcap; ka.sl_j = fa.sl_j; ka.sl_d = sl_d; ka.sl_p = fa.sl_p;
    ka.row_cs = fa.row_cs; ka.row_ce = fa.row_ce; ka.row_begin = fa.row_begin; ka.idx_out = fa.idx_out; ka.dist_out = fa.dist_out;
    wc_fin_rank_kernel<<<(rows + RK_WARPS - 1) / RK_WARPS, RK_WARPS * 32, 0, stream>>>(ka);
    WC_CUDA(cudaGetLastError());
    ctx->timed_mask |= 1u << 10;                           // phase 10: the re-score alone (read on demand)
    ctx->k6_stats_d = big_count;                           // [0] rows passed on, [1] live entries, [2] shortlisted candidates, [3] most live entries of a row
    *launches = 6;                                         // select (warp per row), select (row list), bucket scan, scatter, re-score, rank
    return WC_OK;
}
