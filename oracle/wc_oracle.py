"""TEST INFRASTRUCTURE - CPU oracle for the WISECONDOR within-sample comparison hot path.

This module is a plain numpy *restatement* of the reference's algorithm (not a copy of its code), written
from SURVEY.md section 8(a).  Every function cites the reference lines it follows
(`/root/reference/<file>:<lines>`).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import it; the product (wisecondor_b200/) never does.

PARITY PIN: the reference ships no tests, golden vectors or fixtures (SURVEY.md section 4), so this oracle
is pinned against *outputs of the reference itself run in the build container*: oracle/make_ref.py produces a
mechanically converted Python-3 copy under oracle/_ref/ and tests/test_oracle_vs_ref.py /
tests/golden/make_golden.py compare function by function (bit-exact where the reference is deterministic).
The committed fixtures in tests/golden/ are those reference outputs.  One documented deviation: scikit-learn's
PCA is pinned to svd_solver='full' (today's default picks a randomized, non-deterministic solver - SURVEY.md
section 8(c)); PCA outputs are therefore compared to 1e-9 relative, not bit-exact.
"""
import numpy as np

FILLER_DIST = 1e10          # wisetools.py:306,312 - initial distance / running maximum
FILLER_INDEX = -1           # wisetools.py:305


# --------------------------------------------------------------------------------------------------------
# ingest                                                                        wisetools.py:220-278
# --------------------------------------------------------------------------------------------------------
def scale_sample(sample, from_size, to_size):
    """Down-bin counts by an integer factor (wisetools.py:220-237): out[i] = sum(chrom[i*f:(i+1)*f]),
    new length ceil(len/f).  Identity when sizes agree or to_size is None; non-multiples are an error."""
    if to_size is None or from_size == to_size:
        return sample
    if to_size == 0 or from_size == 0 or to_size < from_size or to_size % from_size > 0:
        raise ValueError("Impossible binsize scaling requested: %s to %s" % (from_size, to_size))
    f = int(to_size // from_size)
    out = {}
    for chrom, data in sample.items():
        if data is None:
            raise TypeError("chromosome %s absent" % chrom)   # the reference raises on len(None) too
        n = int(np.ceil(len(data) / float(f)))
        padded = np.zeros(n * f, dtype=np.int64)
        padded[:len(data)] = data
        out[chrom] = padded.reshape(n, f).sum(axis=1).astype(np.int32)
    return out


def to_numpy_array(samples):
    """Stack chr1..22 of every sample to bins x samples, divide each sample by its total, keep bins whose
    sum over samples is > 0 (wisetools.py:240-264).  Returns (masked N x S, chromBins[22], mask[Nraw])."""
    nsamp = len(samples)
    chrom_bins = []
    blocks = []
    for c in range(1, 23):
        n = max(s[str(c)].shape[0] for s in samples)
        blk = np.zeros((n, nsamp), dtype=float)
        for i, s in enumerate(samples):
            blk[:, i] = s[str(c)]                      # raises when lengths differ, like the reference (:250)
        chrom_bins.append(n)
        blocks.append(blk)
    data = np.concatenate(blocks, axis=0)
    data = data / data.sum(axis=0)                     # :255-256 (sum taken before masking)
    mask = data.sum(axis=1) > 0                        # :259-260
    return data[mask, :], chrom_bins, mask


def to_numpy_ref_format(sample, chrom_bins, mask):
    """Test sample -> masked normalised vector in the reference's bin layout (wisetools.py:267-278):
    zero-pad / truncate each chromosome to chrom_bins[c], divide by the total, apply the mask."""
    parts = []
    for c in range(1, 23):
        want = int(chrom_bins[c - 1])
        v = np.zeros(want, dtype=float)
        have = sample[str(c)]
        n = min(want, len(have))
        v[:n] = have[:n]
        parts.append(v)
    data = np.concatenate(parts)
    data = data / data.sum()
    return data[mask]


# --------------------------------------------------------------------------------------------------------
# PCA                                                                            wisetools.py:89-113
# --------------------------------------------------------------------------------------------------------
def train_pca(masked, ncomp=3):
    """Exact top-`ncomp` principal subspace of the samples x bins matrix and the corrected ratio matrix
    (wisetools.py:89-101 with sklearn PCA(svd_solver='full')).  Returns (corrected N x S, components
    ncomp x N, mean N).  Component signs follow sklearn's svd_flip (largest |entry| of each row of Vt
    positive); they do not affect `corrected`."""
    t = np.ascontiguousarray(masked.T)                 # S x N
    # pca.mean_: scikit-learn reduces the Fortran-ordered view refData.T along its contiguous axis, i.e. each bin's S
    # values with numpy's pairwise sum - the same additions as a row mean of the C-ordered bins x samples matrix
    mean = np.ascontiguousarray(masked).mean(axis=1)
    tc = t - mean
    u, s, vt = np.linalg.svd(tc, full_matrices=False)
    vt = vt[:ncomp]
    signs = np.sign(vt[np.arange(ncomp), np.argmax(np.abs(vt), axis=1)])
    signs[signs == 0] = 1.0
    vt = vt * signs[:, None]
    proj = tc @ vt.T                                   # transform            (:94)
    recon = proj @ vt + mean                           # inverse_transform    (:95)
    corrected = t / recon                              # (:96)
    return corrected.T, vt, mean


def apply_pca(x, mean, components):
    """x / ((x - mean) C^T C + mean)   (wisetools.py:104-113)."""
    proj = np.dot(np.array([x]) - mean, components.T)
    recon = (np.dot(proj, components) + mean)[0]
    return x / recon


# --------------------------------------------------------------------------------------------------------
# reference-bin search                                                         wisetools.py:298-398
# --------------------------------------------------------------------------------------------------------
def get_part(partnum, outof, bincount):
    """Rows of 0-based part `partnum` of `outof` (wisetools.py:358-361)."""
    return int(bincount / float(outof) * partnum), int(bincount / float(outof) * (partnum + 1))


def split_by_chrom(start, end, chrom_bin_sums):
    """Cut [start, end) at chromosome ends -> [chrom, a, b] triples (wisetools.py:340-354).  The first
    triple's `a` may lie before `start`; the caller clamps it (wisetools.py:380-383)."""
    areas = []
    cur = [0, start, 0]
    for i, val in enumerate(chrom_bin_sums):
        cur[0] = i
        if val >= end:
            break
        if start < val < end:
            cur[2] = val
            areas.append(cur)
            cur = [i, val, 0]
        cur[1] = val
    cur[2] = end
    areas.append(cur)
    return areas


def squared_distances_seq(other, row):
    """d_j = sum_s (other[j,s] - row[s])^2 accumulated sequentially over s = 0..S-1 with separately rounded
    subtract, multiply and add - the arithmetic the reference executes at wisetools.py:302 on its
    Fortran-ordered arrays (SURVEY.md 8(a) row 5)."""
    acc = np.zeros(other.shape[0])
    for s in range(other.shape[1]):
        t = other[:, s] - row[s]
        acc = acc + t * t
    return acc


def select_smallest(dist, amount):
    """The reference's streaming insert (wisetools.py:305-321) in closed form: candidates with
    dist < 1e10 (NaN never passes) stably sorted by (dist, index), first `amount`; unfilled slots keep
    index -1 / distance 1e10."""
    idx = np.full(amount, FILLER_INDEX, dtype=np.int32)
    dst = np.full(amount, FILLER_DIST, dtype=np.float64)
    ok = np.flatnonzero(dist < FILLER_DIST)
    order = ok[np.argsort(dist[ok], kind='stable')][:amount]
    idx[:len(order)] = order
    dst[:len(order)] = dist[order]
    return idx, dst


def get_ref_for_bins(amount, start, end, data, other):
    """wisetools.py:298-325 for target rows [start, end) of `data` against candidate rows `other`."""
    idx = np.zeros((end - start, amount), dtype=np.int32)
    dst = np.ones((end - start, amount))
    for t in range(start, end):
        d = squared_distances_seq(other, data[t, :])
        idx[t - start], dst[t - start] = select_smallest(d, amount)
    return idx, dst


def get_reference(corrected, chrom_bins, chrom_bin_sums, amount=100, part=1, parts=1):
    """wisetools.py:364-398: rows of 1-based `part` of `parts`; candidates are all bins of the other
    chromosomes, indexed by their position in that concatenation."""
    n = int(chrom_bin_sums[-1])
    lo, hi = get_part(part - 1, parts, n)
    all_idx, all_dst = [], []
    for chrom, a, b in split_by_chrom(lo, hi, chrom_bin_sums):
        a, b = max(a, lo), min(b, hi)
        cs = int(chrom_bin_sums[chrom] - chrom_bins[chrom])
        ce = int(chrom_bin_sums[chrom])
        other = np.concatenate((corrected[:cs, :], corrected[ce:, :]))
        i, d = get_ref_for_bins(amount, a, b, corrected, other)
        all_idx.extend(i)
        all_dst.extend(d)
    return np.array(all_idx), np.array(all_dst)


# --------------------------------------------------------------------------------------------------------
# within-sample z-scores                                              wisetools.py:328-336, 407-448
# --------------------------------------------------------------------------------------------------------
def get_optimal_cutoff(distances, repeats=3):
    """cut = inf; repeat: cut = mean + 3*std of the distances below cut (wisetools.py:328-336)."""
    cut = float("inf")
    for _ in range(repeats):
        sel = distances[distances < cut]
        cut = np.average(sel) + 3 * np.std(sel)
    return cut


def pairwise_sum(a):
    """numpy's float64 add.reduce over a contiguous 1-D array, restated (the third-party arithmetic behind
    np_mean / np_std / np_sum at wisetools.py:426-427, 471; numpy `pairwise_sum` in loops_utils.h): n < 8
    sequential from 0.0... precisely: n < 8 -> left-to-right sum starting from a[0]'s block; n <= 128 -> eight
    interleaved accumulators combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the n%8 tail added
    sequentially; larger n -> split at n/2 rounded down to a multiple of 8 and recurse.  The CUDA z-score and
    segmentation kernels implement exactly this order; tests pin it against numpy itself."""
    n = len(a)
    if n < 8:
        res = 0.0
        for v in a:
            res = res + float(v)
        return res
    if n <= 128:
        r = [float(a[j]) for j in range(8)]
        i = 8
        while i < n - (n % 8):
            for j in range(8):
                r[j] = r[j] + float(a[i + j])
            i += 8
        res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
        while i < n:
            res = res + float(a[i])
            i += 1
        return res
    n2 = n // 2
    n2 -= n2 % 8
    return pairwise_sum(a[:n2]) + pairwise_sum(a[n2:])


def mean_std_model(a):
    """np.mean / np.std (ddof 0) of a 1-D float64 array in numpy's operation order: mean = pairwise_sum / n;
    std = sqrt(pairwise_sum((a - mean)^2) / n) with separately rounded subtract and multiply."""
    n = len(a)
    m = pairwise_sum(a) / n
    dev = [float(v) - m for v in a]
    sq = [d * d for d in dev]
    return m, float(np.sqrt(pairwise_sum(sq) / n))


def try_sample(test, test_copy, indexes, distances, chrom_bins, chrom_bin_sums, cutoff):
    """One z-score pass (wisetools.py:407-435).  Per bin: reference values = test_copy without the bin's
    own chromosome, gathered at indexes[i][distances[i] < cutoff], negatives dropped; z = (x-mean)/std,
    r = x/mean (numpy mean/std, ddof 0)."""
    n = int(chrom_bin_sums[-1])
    z = np.zeros(n)
    r = np.zeros(n)
    sizes = np.zeros(n)
    sd_sum, sd_num = 0.0, 0
    with np.errstate(all='ignore'):
        for c in range(len(chrom_bins)):
            cs = int(chrom_bin_sums[c] - chrom_bins[c])
            ce = int(chrom_bin_sums[c])
            other = np.concatenate((test_copy[:cs], test_copy[ce:]))
            for i in range(cs, ce):
                ref = other[indexes[i][distances[i] < cutoff]]
                ref = ref[ref >= 0]
                if ref.shape[0] == 0:
                    m = sd = np.nan
                else:
                    m = np.mean(ref)
                    sd = np.std(ref)
                if not np.isnan(sd):
                    sd_sum += sd
                    sd_num += 1
                z[i] = (test[i] - m) / sd
                r[i] = test[i] / m
                sizes[i] = ref.shape[0]
        avg = sd_sum / sd_num if sd_num else np.nan
    return z, r, sizes, avg


def repeat_test(test, indexes, distances, chrom_bins, chrom_bin_sums, cutoff, threshold, repeats):
    """wisetools.py:438-448: `repeats` passes; after each, bins with |z| >= threshold are set to -1 in the
    working copy so they stop serving as reference values.  Returns the last pass."""
    copy = np.copy(test)
    out = None
    for _ in range(repeats):
        out = try_sample(test, copy, indexes, distances, chrom_bins, chrom_bin_sums, cutoff)
        with np.errstate(all='ignore'):
            copy[np.abs(out[0]) >= threshold] = -1
    return out


# --------------------------------------------------------------------------------------------------------
# Stouffer segmentation                              wisetools.py:466-487, triarray.py:13-84
# --------------------------------------------------------------------------------------------------------
def run_value(region, x, y):
    """Triangle entry (x, y): sum(region[x..y]) / sqrt(y-x+1) with numpy's summation (wisetools.py:471)."""
    return np.sum(region[x:y + 1]) / np.sqrt(y - x + 1)


def fill_triangle(region, region_r=None, min_effect=0):
    """Packed row-major upper triangle of run values (wisetools.py:466-487; layout triarray.py:26-29).
    With min_effect != 0 entries whose |median(R[x..y]) - 1| < min_effect are zeroed (fillTriMin)."""
    n = region.shape[0]
    out = np.zeros(n * (n + 1) // 2)
    k = 0
    for x in range(n):
        for y in range(x, n):
            # the reference's own form of the test (wisetools.py:483): a NaN median (a NaN ratio in the run) compares
            # False and zeroes the entry
            if min_effect == 0 or abs(np.median(region_r[x:y + 1]) - 1) >= min_effect:
                out[k] = run_value(region, x, y)
            else:
                out[k] = 0
            k += 1
    return out


def _row_start(n, x):
    return x * n - x * (x - 1) // 2


def _lin_to_xy(n, pos):
    """triarray.py:46-51."""
    edge = n
    while pos >= edge:
        pos -= edge
        edge -= 1
    return n - edge, pos + n - edge


def segment_triangle(tri, n, threshold, min_search=3, lo=0, hi=None):
    """triarray.py:59-84 on the sub-range [lo, hi) of a packed triangle of edge n, without copying
    sub-triangles: the entries of a sub-triangle are the parent's entries (triarray.py:31-38), visited
    in the same row-major order, so first-occurrence argmax/argmin are preserved.  Coordinates returned are
    absolute (the reference's offset bookkeeping at :81 folded in)."""
    if hi is None:
        hi = n
    m = hi - lo
    if m <= 0:
        # an empty TriArr: argmax on an empty array raises in numpy; the driver never builds one
        raise ValueError("empty triangle")
    # row x of the sub-triangle = entries (x, x..hi-1) = the first hi-x entries of the parent's row x
    flat = np.concatenate([tri[_row_start(n, x): _row_start(n, x) + (hi - x)] for x in range(lo, hi)])
    with np.errstate(all='ignore'):
        cpos = int(np.argmax(flat))
        cval = flat[cpos]
        bpos = int(np.argmin(flat))
        bval = flat[bpos]
        if abs(bval) > cval:
            cval, cpos = bval, bpos
        if abs(cval) < threshold:
            return []
    x, y = _lin_to_xy(m, cpos)
    out = []
    if x > min_search:
        out.extend(segment_triangle(tri, n, threshold, min_search, lo, lo + x))
    out.append((cval, (lo + x, lo + y)))
    if y + 1 < m - min_search:
        out.extend(segment_triangle(tri, n, threshold, min_search, lo + y + 1, hi))
    return out


def segment_region(region, threshold, min_search=3, region_r=None, min_effect=0):
    """fillTriMin + chromosome-wide value + segmentTri for one chromosome (wisecondor.py:236-238).
    Returns (chrom_wide_z, [(z, (x, y)), ...]) with inclusive cleaned-bin coordinates."""
    n = region.shape[0]
    tri = fill_triangle(region, region_r, min_effect)
    cw = tri[n - 1]                                    # getValue(0, n-1)
    return cw, segment_triangle(tri, n, threshold, min_search)


def prefix_run_value(prefix, x, y):
    """Relaxed form used for large-shape checks only: (P[y+1]-P[x]) / sqrt(len) - not bit-identical to
    run_value (different summation order), agrees to ~1e-15 relative."""
    return (prefix[y + 1] - prefix[x]) / np.sqrt(y - x + 1)


def segment_region_prefix(region, threshold, min_search=3):
    """Segmentation with prefix-sum run values (vectorised; O(n^2) memory-free per row).  A relaxed oracle for
    chromosome sizes where fill_triangle's Python double loop is out of reach; tests/ pin it against
    segment_region on small cases."""
    n = region.shape[0]
    prefix = np.concatenate(([0.0], np.cumsum(region)))
    inv = 1.0 / np.sqrt(np.arange(1, n + 1, dtype=float))

    def best(lo, hi):
        bmax, bmin = (-np.inf, 0, 0), (np.inf, 0, 0)
        for x in range(lo, hi):
            vals = (prefix[x + 1:hi + 1] - prefix[x]) / np.sqrt(np.arange(1, hi - x + 1, dtype=float))
            j = int(np.argmax(vals))
            if vals[j] > bmax[0]:
                bmax = (vals[j], x, x + j)
            j = int(np.argmin(vals))
            if vals[j] < bmin[0]:
                bmin = (vals[j], x, x + j)
        return bmax, bmin

    def rec(lo, hi):
        bmax, bmin = best(lo, hi)
        cval, x, y = bmax
        if abs(bmin[0]) > cval:
            cval, x, y = bmin
        if abs(cval) < threshold:
            return []
        out = []
        if x - lo > min_search:
            out.extend(rec(lo, x))
        out.append((cval, (x, y)))
        if (y - lo) + 1 < (hi - lo) - min_search:
            out.extend(rec(y + 1, hi))
        return out

    del inv
    cw = (prefix[n] - prefix[0]) / np.sqrt(n)
    return cw, rec(0, n)


def segment_region_exact(region, threshold, min_search=3, max_window=10 ** 6):
    """segment_region's result, bit for bit, for finite z at chromosome sizes (5 000 - 25 000 bins) where
    fill_triangle's O(n^3) loop is out of reach.

    Per pending range [lo, hi) the runs are located with fp64 prefix sums of region[lo:hi] (rebased per range), one
    vectorised row x at a time.  Every run whose located |value| is within `tol` of the located maximum M is kept, with
    tol = 4 m eps sum|region[lo:hi]| + 8 eps M: each prefix end and numpy's own pairwise sum are off by at most
    m eps sum|z|, the subtraction, 1/sqrt and product by a few eps |value|.  Those runs alone are re-scored exactly
    as the reference does (np.sum(region[x:y+1]) / np.sqrt(y-x+1), wisetools.py:471) and the reference's rules decide:
    max, then min, abs(min) > max, first occurrence in row-major order, threshold, recursion (triarray.py:59-84).  A
    window of more than `max_window` runs raises instead of guessing."""
    z = np.asarray(region, dtype=np.float64)
    n = z.shape[0]
    if n == 0:
        raise ValueError("empty region")
    if not np.isfinite(z).all():
        raise ValueError("segment_region_exact takes finite z only")
    eps = np.finfo(np.float64).eps
    inv = 1.0 / np.sqrt(np.arange(1, n + 1, dtype=np.float64))

    def champion(lo, hi):
        m = hi - lo
        p = np.concatenate(([0.0], np.cumsum(z[lo:hi])))
        rowmax = np.empty(m)
        for x in range(m):
            rowmax[x] = np.max(np.abs((p[x + 1:] - p[x]) * inv[:m - x]))
        big = float(np.max(rowmax))
        tol = 4.0 * m * eps * float(np.sum(np.abs(z[lo:hi]))) + 8.0 * eps * big
        if big + tol < threshold:                             # every |value| is below the threshold: no call
            return None
        floor = big - 2.0 * tol
        cands = []
        for x in np.flatnonzero(rowmax >= floor):
            ys = np.flatnonzero(np.abs((p[x + 1:] - p[x]) * inv[:m - x]) >= floor)
            cands.extend((lo + int(x), lo + int(x) + int(j)) for j in ys)
            if len(cands) > max_window:
                raise ValueError("segment_region_exact: more than %d runs within %g of the maximum" % (max_window, tol))
        best_max = best_min = None
        for x, y in cands:                                    # row-major order: strict comparisons keep the first
            v = np.sum(z[x:y + 1]) / np.sqrt(y - x + 1)
            if best_max is None or v > best_max[0]:
                best_max = (v, x, y)
            if best_min is None or v < best_min[0]:
                best_min = (v, x, y)
        return best_min if abs(best_min[0]) > best_max[0] else best_max

    calls = []
    pending = [(0, n)]
    while pending:
        lo, hi = pending.pop()
        best = champion(lo, hi)
        if best is None or abs(best[0]) < threshold:
            continue
        v, x, y = best
        calls.append((v, (x, y)))
        if x - lo > min_search:
            pending.append((lo, x))
        if (y - lo) + 1 < (hi - lo) - min_search:
            pending.append((y + 1, hi))
    calls.sort(key=lambda c: c[1][0])                         # the reference's in-order recursion: left, call, right
    return np.sum(z) / np.sqrt(n), calls


# --------------------------------------------------------------------------------------------------------
# test driver                                                                  wisecondor.py:174-281
# --------------------------------------------------------------------------------------------------------
def inflate(array, mask):
    """wisetools.py:281-288."""
    out = np.zeros(mask.shape[0])
    out[np.asarray(mask, dtype=bool)] = array
    return out


def inflate_multi(array, masks):
    """wisetools.py:291-295."""
    for m in reversed(masks):
        array = inflate(array, m)
    return array


def call_to_raw(seg, chrom, chrom_sizes, shifter_inflated):
    """Cleaned-bin run (x, y) -> raw bin coordinates within the chromosome, reproducing the walk at
    wisecondor.py:241-253 (the end walk restarts on the start bin, so end = raw(y-1)+1 when y > x)."""
    base = int(sum(chrom_sizes[:chrom]))
    pos = base
    filled = 0
    while filled <= seg[0]:
        filled += int(shifter_inflated[pos] != 0)
        pos += 1
    pos -= 1
    end = pos
    while filled <= seg[1]:
        filled += int(shifter_inflated[end] != 0)
        end += 1
    return pos - base, end - base


def test_sample(sample, sample_binsize, ref, minzscore=None, chromosomes=tuple(range(1, 23)), mineffectsize=0,
                multitest=1000, minrefbins=25, repeats=5, segmenter=segment_region):
    """toolTest (wisecondor.py:174-281) as a function: `ref` is a dict with the reference-npz keys.  Returns
    a dict with the result-npz keys (without arguments/runtime)."""
    from scipy.stats import norm
    binsize = ref['binsize']
    indexes, distances = ref['indexes'], ref['distances']
    chrom_sizes, mask = ref['chromosome_sizes'], ref['mask']
    masked_sizes = ref['masked_sizes']
    sums = [int(sum(masked_sizes[:x + 1])) for x in range(len(masked_sizes))]
    sample = scale_sample(sample, sample_binsize, binsize)
    test = to_numpy_ref_format(sample, chrom_sizes, mask)
    test = apply_pca(test, ref['pca_mean'], ref['pca_components'])
    cutoff = get_optimal_cutoff(distances, 3)
    z_thr = norm.ppf(1 - 1. / (sum(masked_sizes) * 0.5 * multitest))
    if minzscore is not None:
        z_thr = minzscore
    z, r, sizes, sd_avg = repeat_test(np.copy(test), indexes, distances, masked_sizes, sums, cutoff, z_thr, repeats)
    keep = sizes >= minrefbins
    cz, cr = z[keep], r[keep]
    csums = [int(np.sum(keep[:v])) for v in sums]
    cbins = [csums[0]] + [csums[i] - csums[i - 1] for i in range(1, len(csums))]
    shifter = inflate_multi(np.ones(cz.shape, dtype=bool), [mask, keep])
    calls, cwz = [], []
    for c in [x - 1 for x in chromosomes]:
        a, b = int(sum(cbins[:c])), int(sum(cbins[:c + 1]))
        if mineffectsize != 0:
            cw, segs = segment_region(cz[a:b], z_thr, 3, cr[a:b], mineffectsize)
        else:
            cw, segs = segmenter(cz[a:b], z_thr, 3)
        cwz.append(cw)
        for val, (x, y) in segs:
            s_raw, e_raw = call_to_raw((x, y), c, chrom_sizes, shifter)
            calls.append([c + 1, s_raw, e_raw, val, np.median(cr[a + x:a + y + 1]) - 1])
    iz = inflate_multi(cz, [mask, keep])
    ir = inflate_multi(cr - 1, [mask, keep])
    res_z, res_r = [], []
    for c in range(len(chrom_sizes)):
        a, b = int(sum(chrom_sizes[:c])), int(sum(chrom_sizes[:c + 1]))
        res_z.append(iz[a:b])
        res_r.append(ir[a:b])
    return dict(binsize=binsize, results_r=res_r, results_z=res_z, results_cwz=np.array(cwz),
                results_calls=np.array(calls), threshold_z=z_thr, asdef=sd_avg, aasdef=sd_avg * z_thr,
                _z=z, _r=r, _sizes=sizes, _cutoff=cutoff, _test=test)
