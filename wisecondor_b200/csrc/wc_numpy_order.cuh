// wisecondor_b200 - numpy's float64 summation order on the device.
//
// The reference calls np_sum / np_mean / np_std on small contiguous 1-D arrays (wisetools.py:426-427 reference
// values of a bin, :471 z-scores of a run).  numpy reduces those with its pairwise scheme (third-party code, numpy
// `pairwise_sum`): fewer than 8 elements are added left to right; up to 128 elements go through eight interleaved
// accumulators r[j] += a[i + j] that are combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) before the n % 8 tail is
// added left to right; longer arrays are split at n/2 rounded down to a multiple of 8 and the halves' sums added.
// Reproducing that order makes the z-scores and run values bit-identical to the reference's at no extra cost.
// oracle/wc_oracle.py:pairwise_sum is the same statement in Python, pinned against numpy itself by the tests.
#pragma once

// One thread sums f(0..n-1), n <= 128.  `f` returns the i-th element (any separately rounded expression).
template <class F>
__device__ __forceinline__ double np_sum_leaf(F f, int n) {
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = __dadd_rn(res, f(i));
        return res;
    }
    double r0 = f(0), r1 = f(1), r2 = f(2), r3 = f(3), r4 = f(4), r5 = f(5), r6 = f(6), r7 = f(7);
    const int full = n - (n & 7);
    int i = 8;
    for (; i < full; i += 8) {
        r0 = __dadd_rn(r0, f(i));
        r1 = __dadd_rn(r1, f(i + 1));
        r2 = __dadd_rn(r2, f(i + 2));
        r3 = __dadd_rn(r3, f(i + 3));
        r4 = __dadd_rn(r4, f(i + 4));
        r5 = __dadd_rn(r5, f(i + 5));
        r6 = __dadd_rn(r6, f(i + 6));
        r7 = __dadd_rn(r7, f(i + 7));
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r0, r1), __dadd_rn(r2, r3)), __dadd_rn(__dadd_rn(r4, r5), __dadd_rn(r6, r7)));
    for (; i < n; ++i) res = __dadd_rn(res, f(i));
    return res;
}

// One thread sums f(0..n-1) for any n: numpy's recursion, unrolled with an explicit stack of pending right halves.
// (n <= 128 * 2^24; depth of the stack = number of halvings.)
template <class F>
__device__ __forceinline__ double np_sum_thread(F f, int n) {
    if (n <= 128) return np_sum_leaf(f, n);
    // Post-order evaluation of the split tree: `val[d]` holds the finished left sum waiting at depth d.
    int off_stack[26], len_stack[26];
    double val[26];
    unsigned char state[26];          // 0 = left child pending, 1 = right child pending
    int sp = 0;
    off_stack[0] = 0; len_stack[0] = n; state[0] = 0;
    double ret = 0.0;
    while (sp >= 0) {
        const int off = off_stack[sp], len = len_stack[sp];
        if (len <= 128) {
            ret = np_sum_leaf([&](int i) { return f(off + i); }, len);
            --sp;
            continue;
        }
        int n2 = len / 2;
        n2 -= n2 & 7;
        if (state[sp] == 0) {
            state[sp] = 1;
            ++sp;
            off_stack[sp] = off; len_stack[sp] = n2; state[sp] = 0;
        } else if (state[sp] == 1) {
            val[sp] = ret;             // left sum done
            state[sp] = 2;
            ++sp;
            off_stack[sp] = off + n2; len_stack[sp] = len - n2; state[sp] = 0;
        } else {
            ret = __dadd_rn(val[sp], ret);
            --sp;
        }
    }
    return ret;
}

// The same order, fed one element at a time: begin(n) fixes the split tree of n elements, push() takes them in index
// order, and after the n-th push `res` holds the sum.  The caller needs no storage for the elements, so it can drop
// values on the fly (numpy sums the compacted array: the tree is that of the kept count).  The stack holds, per
// ancestor of the current leaf, either the pending right half's length or the finished left half's sum; it is touched
// once per leaf (>= 64 elements).  The leaf's eight accumulators form a ring that rotates by one per element, so
// r0 always receives element p, without run-time register indexing; `full` is a multiple of 8, so the ring is back in
// place when the accumulators are combined.
constexpr int NP_STREAM_DEPTH = 26;    // n <= 128 * 2^24 as above
struct NpStream {
    double r0, r1, r2, r3, r4, r5, r6, r7, res;
    int leaf, p, full, d;                      // current leaf's length, position in it, 8-multiple part; frames
    int rlen[NP_STREAM_DEPTH];                 // > 0: left half in progress, right half of this length pending
    double lsum[NP_STREAM_DEPTH];              // right half in progress: the left half's sum

    __device__ __forceinline__ void descend(int len) {       // start the leftmost leaf of a piece of len elements
        while (len > 128) {
            int h = len / 2;
            h -= h & 7;
            rlen[d] = len - h;
            ++d;
            len = h;
        }
        leaf = len; p = 0; full = len - (len & 7); res = 0.0;
    }
    __device__ __forceinline__ void begin(int n) { d = 0; descend(n); }    // n == 0: res = 0.0 at once

    __device__ __forceinline__ void push(double v) {
        if (p < full) {
            const double t = p < 8 ? v : __dadd_rn(r0, v);
            r0 = r1; r1 = r2; r2 = r3; r3 = r4; r4 = r5; r5 = r6; r6 = r7; r7 = t;
            if (p + 1 == full)
                res = __dadd_rn(__dadd_rn(__dadd_rn(r0, r1), __dadd_rn(r2, r3)), __dadd_rn(__dadd_rn(r4, r5), __dadd_rn(r6, r7)));
        } else {
            res = __dadd_rn(res, v);                              // n < 8, or the n % 8 tail
        }
        if (++p == leaf) finish_leaf();
    }
    __device__ __forceinline__ void finish_leaf() {
        double s = res;
        while (d > 0) {
            const int f = d - 1;
            if (rlen[f] > 0) {                                    // a left half is done: start its right sibling
                lsum[f] = s;
                const int len = rlen[f];
                rlen[f] = 0;
                descend(len);
                return;
            }
            s = __dadd_rn(lsum[f], s);                            // a right half is done: (left + right) goes up
            d = f;
        }
        res = s;
        leaf = -1;                                                // finished: further pushes are a caller error
    }
};
