// wisecondor_b200 - wide-refsize reference-bin search (wc_newref_topk_wide): refsize up to WC_WIDE_REFSIZE_MAX.
// Textually included by wc_search.cu after the narrow search.  Shares no kernel with it: every launch of
// wc_newref_topk is unchanged.
//
// The narrow search bounds every row's candidates by a streaming filter whose buffers, shortlists and rank are sized for
// k <= 384.  Here every distance of a chunk of target rows is computed exactly and kept:
//   K5w wc_wide_dist_kernel  exact fp64 distances of R target rows x all N bins, in the reference's operation order
//                            (sequential over samples, separately rounded subtract / multiply / add, as K6b), tiled 64 x 64
//                            so each operand row is read once per tile from L2; own-chromosome columns and d >= 1e10 / NaN
//                            are stored as +inf                                                   (FP64 bound)
//   K6w wc_wide_rank_kernel  one CTA per row: radix select of the k-th smallest (distance, bin) pair on the distances' bit
//                            patterns (non-negative doubles: unsigned order == value order), the <= k winners gathered into
//                            shared memory, bitonic sort by (distance, bin), remap to other-chromosome coordinates, fillers
// The values are final, so there is no filter margin, no re-score and no exhaustive fallback: the result is exact by
// construction.  D[R][N] is the chunk buffer; R is a multiple of 128 chosen from WIDE_CHUNK_BYTES.
#pragma once

constexpr int WIDE_TILE = 64;                  // K5w: target rows x bins per CTA
constexpr int WIDE_SK = 16;                    // K5w: samples staged per step
constexpr int WIDE_DIST_THREADS = 256;         // 16 x 16 threads, 4 x 4 entries each
constexpr int WIDE_RANK_THREADS = 512;
constexpr size_t WIDE_CHUNK_BYTES = (size_t)1 << 30;   // D of one chunk: 2 304 rows at 50 kb (N = 57 633)
constexpr u64 WIDE_KEY_NONE = 0x7ff0000000000000ull;    // bits of +inf: not a candidate

__global__ void __launch_bounds__(WIDE_DIST_THREADS) wc_wide_dist_kernel(const double* __restrict__ X, int N, int S, int row0,
                                                                         int rows, const int* __restrict__ row_cs,
                                                                         const int* __restrict__ row_ce, double* __restrict__ D) {
    __shared__ double sA[WIDE_SK][WIDE_TILE + 1];      // target rows, sample-major
    __shared__ double sB[WIDE_SK][WIDE_TILE + 1];      // candidate bins, sample-major
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int cb = blockIdx.x * WIDE_TILE, rb = blockIdx.y * WIDE_TILE;   // first bin, first local row of the tile
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    const int ls = tid & 15, lr = tid >> 4;            // loader: sample ls of rows lr, lr + 16, ...
    for (int s0 = 0; s0 < S; s0 += WIDE_SK) {
        const int s = s0 + ls;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int r = lr + 16 * q;
            const int ra = rb + r, rc = cb + r;
            sA[ls][r] = (ra < rows && s < S) ? __ldg(X + (size_t)(row0 + ra) * S + s) : 0.0;
            sB[ls][r] = (rc < N && s < S) ? __ldg(X + (size_t)rc * S + s) : 0.0;
        }
        __syncthreads();
        const int ns = S - s0 < WIDE_SK ? S - s0 : WIDE_SK;
        for (int t = 0; t < ns; ++t) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = sA[t][ty + 16 * i]; b[i] = sB[t][tx + 16 * i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const double v = __dsub_rn(b[j], a[i]);          // (x_j[s] - x_row[s]): K6b's operand order
                    acc[i][j] = __dadd_rn(acc[i][j], __dmul_rn(v, v));
                }
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int rl = rb + ty + 16 * i;
        if (rl >= rows) continue;
        const int cs = row_cs[row0 + rl], ce = row_ce[row0 + rl];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = cb + tx + 16 * j;
            if (c >= N) continue;
            double d = acc[i][j];
            if ((c >= cs && c < ce) || !(d < 1e10)) d = INFINITY;    // the reference's 1e10 cut; NaN never passes
            D[(size_t)rl * N + c] = d;
        }
    }
}

// The r-th smallest (1-based) of the keys of the columns j < N for which key(j, kv) returns true: MSB-first radix select in
// 8-bit digits from bit `top`; counts are warp-aggregated before the shared-memory atomics (the first digits of a row's
// keys are nearly all equal).  Returns the key; *s_r = its rank among the keys equal to it, *s_eq = how many keys equal it.
template <typename Key>
__device__ u64 wide_radix_select(Key key, int N, int r, int top, unsigned* hist, u64* s_prefix, int* s_r, int* s_eq) {
    const int tid = threadIdx.x, lane = tid & 31;
    u64 prefix = 0ull, mask = 0ull;
    for (int shift = top; shift >= 0; shift -= 8) {
        for (int b = tid; b < 256; b += blockDim.x) hist[b] = 0u;
        __syncthreads();
        const int jend = (N + 31) / 32 * 32;
        for (int j = tid; j < jend; j += blockDim.x) {
            u64 kv = 0ull;
            const bool ok = j < N && key(j, kv) && (kv & mask) == prefix;
            const unsigned dig = ok ? (unsigned)((kv >> shift) & 255u) : 256u;
            const unsigned peers = __match_any_sync(0xffffffffu, dig);
            if (ok && lane == __ffs(peers) - 1) atomicAdd(hist + dig, (unsigned)__popc(peers));
        }
        __syncthreads();
        if (tid == 0) {
            unsigned cum = 0u;
            int sel = 255;
            for (int b = 0; b < 256; ++b) {
                if (cum + hist[b] >= (unsigned)r) { sel = b; break; }
                cum += hist[b];
            }
            r -= (int)cum;
            *s_eq = (int)hist[sel];
            prefix |= (u64)sel << shift;
            *s_prefix = prefix;
            *s_r = r;
        }
        __syncthreads();
        prefix = *s_prefix;
        r = *s_r;
        mask |= 255ull << shift;
        __syncthreads();
    }
    return prefix;
}

struct WideRankArgs {
    const double* D;       // [rows][N] of this chunk
    int N, k, row0;        // row0: global bin of the chunk's first row
    const int* row_cs;
    const int* row_ce;
    int32_t* idx_out;      // [rows][k] of this chunk
    double* dist_out;
};

__global__ void __launch_bounds__(WIDE_RANK_THREADS) wc_wide_rank_kernel(const WideRankArgs a) {
    extern __shared__ __align__(16) unsigned char wide_raw[];
    __shared__ unsigned hist[256];
    __shared__ u64 s_prefix;
    __shared__ int s_r, s_eq, s_n, s_total;
    const int tid = threadIdx.x;
    const int rl = blockIdx.x, row = a.row0 + rl;
    const int cs = a.row_cs[row], ce = a.row_ce[row];
    const u64* drow = reinterpret_cast<const u64*>(a.D + (size_t)rl * a.N);
    int32_t* out_i = a.idx_out + (size_t)rl * a.k;
    double* out_d = a.dist_out + (size_t)rl * a.k;

    // candidates: every stored value below +inf (K5w stored +inf for the excluded ones)
    if (tid == 0) { s_total = 0; s_n = 0; }
    __syncthreads();
    int cnt = 0;
    for (int j = tid; j < a.N; j += blockDim.x) cnt += drow[j] < WIDE_KEY_NONE ? 1 : 0;
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((tid & 31) == 0) atomicAdd(&s_total, cnt);
    __syncthreads();
    const int need = s_total < a.k ? s_total : a.k;

    u64 T = WIDE_KEY_NONE;                  // the need-th smallest distance key
    int J = 0x7fffffff;                     // among keys == T, bins <= J are taken
    if (need > 0) {
        auto dkey = [&](int j, u64& kv) { kv = drow[j]; return kv < WIDE_KEY_NONE; };
        T = wide_radix_select(dkey, a.N, need, 56, hist, &s_prefix, &s_r, &s_eq);
        const int r_eq = s_r, n_eq = s_eq;
        if (n_eq > r_eq) {                  // a tie at the k-th place: the r_eq smallest bins among the equal keys
            auto jkey = [&](int j, u64& kv) { kv = (u64)j; return drow[j] == T; };
            J = (int)wide_radix_select(jkey, a.N, r_eq, 24, hist, &s_prefix, &s_r, &s_eq);
        }
    }
    // gather the winners (exactly `need` of them) and sort them by (distance, bin)
    int P = 32;
    while (P < need) P <<= 1;
    u64* sk = reinterpret_cast<u64*>(wide_raw);
    int* sj = reinterpret_cast<int*>(sk + P);
    for (int e = tid; e < P; e += blockDim.x) { sk[e] = ~0ull; sj[e] = 0x7fffffff; }
    __syncthreads();
    if (need > 0) {
        for (int j = tid; j < a.N; j += blockDim.x) {
            const u64 kv = drow[j];
            if (kv < T || (kv == T && j <= J)) {
                const int p = atomicAdd(&s_n, 1);
                if (p < P) { sk[p] = kv; sj[p] = j; }
            }
        }
    }
    __syncthreads();
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = tid; i < P / 2; i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool up = (lo & size) == 0;
                const u64 klo = sk[lo], khi = sk[hi];
                const int jlo = sj[lo], jhi = sj[hi];
                const bool hi_first = khi < klo || (khi == klo && jhi < jlo);
                if (hi_first == up) { sk[lo] = khi; sk[hi] = klo; sj[lo] = jhi; sj[hi] = jlo; }
            }
            __syncthreads();
        }
    }
    for (int t = tid; t < a.k; t += blockDim.x) {
        if (t < need) {
            const int j = sj[t];
            out_i[t] = j >= ce ? j - (ce - cs) : j;
            out_d[t] = __longlong_as_double((long long)sk[t]);
        } else {
            out_i[t] = -1;
            out_d[t] = 1e10;
        }
    }
}
