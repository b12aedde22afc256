"""Adversarial inputs of the reference-bin search (K4h / K5t / K6) and a CPU check that every family has the property it
claims.  The search is a filter followed by an exact re-score; its result is exact only if the filter's margins, K6a''s
histogram select, the shortlist and buffer caps and the fallbacks are right.  Each generator is seeded and names the
branch it aims at; tests/test_search_edges_gpu.py runs them against the C oracle on the GPU.  Here, without a GPU, the
families are held to their claims, so that a GPU pass means what it says."""
import math

import numpy as np
import pytest

import wc_oracle
from wisecondor_b200 import synth

K = 100                                                       # refsize of the families unless stated
MID_BINS = [int(b) for b in np.array(synth.chrom_bins(250000)) // 3]      # N = 3838: whole-matrix calls are symmetric
TC_PIVOTS = 512                                               # wc_search_tc.cuh: pivots of the K5t pivot pass
FP16_LIMIT = 60000.0                                          # K4h: |x - 1| or n / 2 above this -> the fp64 filter


def eps16(S, tc=True):
    """A-priori relative error of the fp16 filter (wc_search.cu, `eps16`): |d~ - d| <= eps16 * (n_i + n_j) + sub."""
    ldh = (S + 4 + 63) // 64 * 64 if tc else (S + 63) // 64 * 64
    return 2.0 ** -10 * (1 + 2.0 ** -11) + (2.0 if tc else 1.0) * ldh * 2.0 ** -23 + (2.0 ** -20 if tc else 2.0 ** -21)


def filter_sub(S, nmax):
    """The subnormal / norm-split term of the fp16 filter's error (the second summand of `filt_madd`)."""
    return 2.0 ** -20 * math.sqrt(S * nmax)


def filt_madd(S, nmax, tc=True):
    """The window every row's threshold is widened by under the fp16 filter (wc_search.cu, `filt_madd`)."""
    return 2.0 * eps16(S, tc) * nmax + filter_sub(S, nmax)


def norms(X):
    xc = X - 1.0
    return (xc * xc).sum(axis=1)


def chrom_of(bins):
    return np.repeat(np.arange(len(bins)), bins)


def other_rows(bins, row):
    """Candidate rows of a target row: every bin of the other chromosomes (wisetools.py:381-383)."""
    c = chrom_of(bins)
    return np.flatnonzero(c != c[row])


def exact_row(X, bins, row):
    """(candidate rows, exact distances in the reference's order) of one target row."""
    cand = other_rows(bins, row)
    return cand, wc_oracle.squared_distances_seq(X[cand], X[row])


def _case(name, X, bins, k=K, **meta):
    return dict(name=name, X=np.ascontiguousarray(X), bins=[int(b) for b in bins], k=int(k), **meta)


# ---------------------------------------------------------------------------------------------------------------------
# families
# ---------------------------------------------------------------------------------------------------------------------
def plain(S=64, k=K, seed=0, bins=None):
    """Benign i.i.d. noise around 1 with bin families (synth.corrected_like): the control every margin is tuned on."""
    bins = list(MID_BINS if bins is None else bins)
    return _case("plain_S%d" % S, synth.corrected_like(bins, S, seed=seed), bins, k)


def near_tie(M, delta, S=64, k=K, seed=0, bins=None, chrom=0):
    """Filter margins and K6a''s histogram select: M near-copies of one low-norm row, spread by delta * |x - 1|, sit on
    chromosome 1 - they are the M nearest bins of every row of the other chromosomes, with distances far closer together
    than the fp16 filter's error, so the k-th and (k+1)-th distances of those rows fall inside the filter's window and
    only the exact re-score can order them.  M around k puts the boundary at the cluster's edge or inside it.  `chrom`
    moves the cluster to another chromosome."""
    bins = list(MID_BINS if bins is None else bins)
    rng = np.random.default_rng(seed + 1)
    X = 1.0 + rng.normal(0.0, 0.05, size=(sum(bins), S))      # i.i.d.: no bin family comes as close as the cluster
    base = 1.0 + rng.normal(0.0, 0.005, S)
    rows = int(sum(bins[:chrom])) + np.sort(rng.choice(bins[chrom], M, replace=False))
    X[rows] = base + delta * np.abs(base - 1.0) * rng.standard_normal((M, S))
    return _case("near_tie_M%d_d%.0e" % (M, delta), X, bins, k, cluster=rows)


def tie_shell(S=64, k=40, plateaus=(39, 40, 41, 80, 120), seed=0):
    """Tie order without duplicate rows (K6d's (distance, bin) compare, the select's equal keys): target p on chromosome
    22 has a shell of plateaus[p] rows x_t +- a e_s (a = 2^-6, one sample each) on chromosome p + 1.  x_t lies on a 2^-10
    grid, so every shell row is at distance a^2 exactly - in fp64 and in fp16 alike - while no two shell rows are equal.
    Plateaus from k - 1 to 3k make the result depend on ordering ties by index."""
    bins = list(MID_BINS)
    X = synth.corrected_like(bins, S, seed=seed)
    rng = np.random.default_rng(seed + 7)
    sums = np.cumsum(bins)
    a = 2.0 ** -6
    targets, shells = [], []
    for p, P in enumerate(plateaus):
        assert P <= 2 * S and P <= bins[p]
        t = int(sums[20]) + 3 + 5 * p                                     # chromosome 22
        X[t] = 1.0 + np.round(rng.normal(0.0, 0.05, S) * 1024) / 1024
        rows = int(sums[p] - bins[p]) + np.sort(rng.choice(bins[p], P, replace=False))
        which = rng.choice(2 * S, P, replace=False)
        for r, w in zip(rows, which):
            X[r] = X[t]
            X[r, w % S] += a if w < S else -a
        targets.append(t)
        shells.append(rows)
    return _case("tie_shell", X, bins, k, targets=targets, shells=shells, tie=a * a)


def sigma_mix(S=64, k=K, seed=0):
    """Skewed norms across chromosomes (K5t's per-row thresholds, the window's n_i term): chromosomes with sigma = 0.005,
    0.05 and 0.5 in turn - norms span four orders of magnitude and the low-sigma bins are everybody's nearest."""
    bins = list(MID_BINS)
    sig = [(0.005, 0.05, 0.5)[c % 3] for c in range(len(bins))]
    X = np.concatenate([synth.corrected_like([b], S, seed=seed + c, sigma=s) for c, (b, s) in enumerate(zip(bins, sig))])
    return _case("sigma_mix", X, bins, k, sigma=sig)


# n = sum of squares, all exact in fp64 whatever the order: 59 999, 60 000 and 60 001 for n / 2
_EDGE_SQUARES = {"below": [300.0, 100.0, 100.0, 99.0, 14.0, 1.0], "at": [300.0, 100.0, 100.0, 100.0],
                 "above": [300.0, 100.0, 100.0, 100.0, 1.0, 1.0]}


def fp16_edge(side, S=64, k=K, seed=0):
    """K4h's range check: one row with n / 2 = 59 999, 60 000 or 60 001 exactly (every |x - 1| <= 300).  The tcgen05 path
    keeps the fp16 filter up to n / 2 = 60 000 and repeats the call with the fp64 filter above it; side 'value' instead
    puts one |x - 1| = 60 001 in a row, which sends every fp16 path to the fp64 filter."""
    bins = list(MID_BINS)
    X = synth.corrected_like(bins, S, seed=seed)
    r = 1000
    X[r] = 1.0
    if side == "value":
        X[r, 5] = 1.0 + 60001.0
    else:
        X[r, :len(_EDGE_SQUARES[side])] = 1.0 + np.array(_EDGE_SQUARES[side])
    return _case("fp16_edge_%s" % side, X, bins, k, row=r, side=side)


def sparse_rows(S=64, k=K, seed=0, count=20):
    """A reference mask keeps any bin where one sample has a read: after the PCA such a bin is ~0 in every sample but
    one, where it is ~1e2.  `count` such rows (|x - 1| up to 141) make n_max / 2 ~ 1e4: still inside fp16's range, but
    filt_madd = 2 eps16 n_max + ... is ~40, far above a normal row's k-th distance - every row's window admits nearly
    every candidate, and the shortlist caps send the rows to the exhaustive fallback K6b."""
    bins = list(MID_BINS)
    X = synth.corrected_like(bins, S, seed=seed)
    rng = np.random.default_rng(seed + 3)
    rows = np.sort(rng.choice(X.shape[0], count, replace=False))
    X[rows] = rng.uniform(0.0, 0.02, size=(count, S))
    X[rows, rng.integers(0, S, count)] = 142.0 * rng.choice([1.0 / 3, 2.0 / 3, 1.0], count)
    X[rows[0], 0] = 142.0
    return _case("sparse_rows", X, bins, k, rows=rows)


def pivot_starved(S=64, k=K, seed=0, zero_rows=0):
    """K5t's pivot pass: the TC_PIVOTS bins of smallest norm all lie on chromosome 1 (700 bins at sigma 0.005), so the
    pivots give its rows no threshold (a row's own chromosome is excluded) and they start the sweep from the initial
    one.  zero_rows > 0 adds a chromosome of rows exactly 1.0 (zero vectors): they tie with each other at distance n_i
    from every other bin - a plateau of exact duplicates for every row."""
    bins = [700] + list(MID_BINS[1:])
    X = np.concatenate([synth.corrected_like([bins[0]], S, seed=seed + 1, sigma=0.005),
                        synth.corrected_like(bins[1:], S, seed=seed)])
    if zero_rows:
        bins.append(zero_rows)
        X = np.concatenate([X, np.ones((zero_rows, S))])
    return _case("pivot_starved" + ("_zero%d" % zero_rows if zero_rows else ""), X, bins, k, zero_rows=zero_rows)


def low_rank(rank, S=64, k=K, seed=0):
    """Distances concentrate: 1 + F G of rank 3-5 plus 1e-4 noise - many candidates lie inside the window around every
    row's k-th distance, the shortlists fill up and the select's fine histogram level decides."""
    bins = list(MID_BINS)
    rng = np.random.default_rng(seed)
    n = sum(bins)
    F = rng.normal(0.0, 0.05, size=(n, rank))
    G = rng.normal(0.0, 1.0, size=(rank, S))
    X = 1.0 + F @ G + rng.normal(0.0, 1e-4, size=(n, S))
    return _case("low_rank_%d" % rank, X, bins, k, rank=rank)


def range_boundary(S):
    """The 1e10 cut (wisetools.py:312-314; K6d, the fused K6 and K6b): only d < 1e10 may enter.  |x - 1| = 1e5 is outside
    fp16's range, so every filter option runs the fp64 filter.  Each target row t (chromosome 1) has candidates
    (chromosome 2) at distance exactly 1e10 and at the nearest doubles on either side: with S >= 3 the next double below
    and above (two 2^-10 steps first, then a, in the reference's summation order); with S = 1 a distance is one rounded
    square and the closest a square of a double gets to 1e10 is two steps away.  Chromosome 3 holds -0.0, exactly 1,
    NaN, +inf and -inf in one sample, and ordinary rows."""
    rng = np.random.default_rng(S)
    lo, hi = np.nextafter(1e10, 0.0), np.nextafter(1e10, np.inf)
    nt = 8
    X = 1.0 + np.round(rng.normal(0.0, 0.05, size=(nt, S)) * 2 ** 20) / 2 ** 20
    steps = []
    if S >= 3:
        a_lo = 1e5
        while a_lo * a_lo != lo - 2.0 ** -19:                 # fl(a^2) = 1e10 - 2 ulp; + 2^-19 -> the next double below
            a_lo = np.nextafter(a_lo, 0.0)
        steps = [(0.0, 1e5), (2.0 ** -10, a_lo), (2.0 ** -10, 1e5)]                # 1e10, below, above (1e10 + 2^-19)
    else:
        below = above = 1e5
        while below * below >= lo:
            below = np.nextafter(below, 0.0)
        while above * above <= hi:
            above = np.nextafter(above, np.inf)
        steps = [(0.0, 1e5), (0.0, below), (0.0, above)]
    cand = []
    for t in range(nt):
        for small, big in steps:
            row = X[t].copy()
            if S >= 3:
                row[0] += small
                row[1] += small
                row[2] += big
            else:
                row[0] += big
            cand.append(row)
    specials = np.ones((10, S)) + rng.normal(0.0, 0.05, size=(10, S))
    specials[0, 0] = -0.0
    specials[1, 0] = 1.0
    specials[2, 0] = np.nan
    specials[3, 0] = np.inf
    specials[4, 0] = -np.inf
    X = np.concatenate([X, np.array(cand), specials])
    bins = [nt, len(cand), 10]
    return _case("range_boundary_S%d" % S, X, bins, k=len(cand) + 12, steps=len(steps))


def pca_counts(binsize, S, sparse, seed=1):
    """PCA-corrected references: synth.bin_model + sample_counts (sample-major int32 counts, chromosome sizes).  With
    `sparse`, 20 bins that are empty in every sample get 1-3 reads in a single sample, so the mask keeps them."""
    bins, lam, fac = synth.bin_model(binsize, bin_seed=seed)
    counts = synth.sample_counts(S, lam, fac, seed=seed + 1)
    if sparse:
        rng = np.random.default_rng(seed + 2)
        empty = np.flatnonzero(counts.sum(axis=0) == 0)
        pick = rng.choice(empty, 20, replace=False)
        counts[rng.integers(0, S, 20), pick] = rng.integers(1, 4, 20)
    return counts, bins


def masked_sizes(bins, mask):
    ends = np.cumsum(bins)
    return [int(mask[e - b:e].sum()) for b, e in zip(bins, ends)]


# The families the GPU parity runs under every filter / select option (the PCA matrices have their own tests)
FAMILIES = {
    "plain": lambda: plain(),
    **{"near_tie_M%d_d%.0e" % (M, d): (lambda M=M, d=d: near_tie(M, d))
       for M in (K - 1, K, K + 1, 2 * K, 3 * K) for d in (1e-3, 1e-5, 1e-7, 1e-9)},
    "tie_shell": lambda: tie_shell(),
    "sigma_mix": lambda: sigma_mix(),
    **{"fp16_edge_%s" % s: (lambda s=s: fp16_edge(s)) for s in ("below", "at", "above", "value")},
    "sparse_rows": lambda: sparse_rows(),
    "pivot_starved": lambda: pivot_starved(),
    "pivot_starved_zero": lambda: pivot_starved(zero_rows=150),
    "low_rank_3": lambda: low_rank(3),
    "low_rank_5": lambda: low_rank(5),
    "range_boundary_S1": lambda: range_boundary(1),
    "range_boundary_S8": lambda: range_boundary(8),
}
# families whose rows DESIGN claims never need the exhaustive fallback at refsize 100
NO_FALLBACK = ("plain",)


# ---------------------------------------------------------------------------------------------------------------------
# CPU checks of the claimed properties
# ---------------------------------------------------------------------------------------------------------------------
def _sample_targets(case, n, seed=0, exclude_chrom=None):
    rng = np.random.default_rng(seed)
    c = chrom_of(case["bins"])
    ok = np.flatnonzero(c != exclude_chrom) if exclude_chrom is not None else np.arange(len(c))
    return rng.choice(ok, n, replace=False)


@pytest.mark.parametrize("M", [K - 1, K, K + 1, 2 * K, 3 * K])
@pytest.mark.parametrize("delta", [1e-3, 1e-5, 1e-7, 1e-9])
def test_near_tie_cluster_is_the_nearest_set_and_inside_the_filter_window(M, delta):
    case = near_tie(M, delta)
    X, bins, k, cl = case["X"], case["bins"], case["k"], case["cluster"]
    assert len(np.unique(X[cl], axis=0)) == M                            # near-copies, never duplicates
    nrm = norms(X)
    e = eps16(X.shape[1])
    exact = 0
    for t in _sample_targets(case, 30, exclude_chrom=0):
        cand, d = exact_row(X, bins, t)
        order = np.lexsort((cand, d))
        assert set(cl) <= set(cand[order[:M + 5]])                        # the cluster is (nearly) the M nearest
        exact += set(cand[order[:M]]) == set(cl)
        dc = d[np.searchsorted(cand, cl)]
        window = e * (nrm[t] + nrm[cl].min())
        assert dc.max() - dc.min() < window                               # the filter cannot order them
        if M > k:
            assert d[order[k]] - d[order[k - 1]] < window                 # the k-th / (k+1)-th gap lies inside it
        assert dc.max() > dc.min()                                        # ... but the exact distances differ
    assert exact >= 20


def test_tie_shells_are_bit_equal_distances_of_distinct_rows():
    case = tie_shell()
    X, bins, k = case["X"], case["bins"], case["k"]
    assert min(len(s) for s in case["shells"]) == k - 1 and max(len(s) for s in case["shells"]) == 3 * k
    for t, rows in zip(case["targets"], case["shells"]):
        d = wc_oracle.squared_distances_seq(X[rows], X[t])
        assert (d == case["tie"]).all()                                   # identical bits
        assert len(np.unique(X[rows], axis=0)) == len(rows)               # distinct rows
        cand, dall = exact_row(X, bins, t)
        assert np.sort(dall)[len(rows)] > case["tie"]                     # the plateau is the nearest set
        xh = (X[rows] - 1.0).astype(np.float16).astype(np.float64)        # fp16 operands are exact: the filter ties too
        assert np.array_equal(xh, X[rows] - 1.0)


def test_sigma_mix_spans_four_orders_of_norm():
    case = sigma_mix()
    nrm = norms(case["X"])
    c = chrom_of(case["bins"])
    med = [np.median(nrm[c == i]) for i in range(3)]
    assert med[0] * 50 < med[1] and med[1] * 50 < med[2]


@pytest.mark.parametrize("side,half_norm", [("below", 59999.0), ("at", 60000.0), ("above", 60001.0)])
def test_fp16_edge_rows_straddle_the_range_limit(side, half_norm):
    case = fp16_edge(side)
    X, r = case["X"], case["row"]
    v = X[r] - 1.0
    assert np.abs(v).max() <= 300.0
    for order in (np.arange(v.size), np.arange(v.size)[::-1]):           # exact in any summation order
        acc = 0.0
        for s in order:
            acc += v[s] * v[s]
        assert acc / 2 == half_norm
    others = np.delete(norms(X), r)
    assert others.max() / 2 < FP16_LIMIT / 1000
    assert np.abs(fp16_edge("value")["X"] - 1.0).max() == FP16_LIMIT + 1


def test_sparse_rows_widen_every_window_beyond_every_row():
    case = sparse_rows()
    X, bins, k = case["X"], case["bins"], case["k"]
    S = X.shape[1]
    nrm = norms(X)
    assert np.abs(X - 1.0).max() == 141.0 and nrm.max() / 2 < FP16_LIMIT     # the fp16 filter still runs
    madd = filt_madd(S, nrm.max())
    kth = []
    for t in _sample_targets(case, 20, seed=1):
        cand, d = exact_row(X, bins, t)
        kth.append(np.sort(d)[k - 1])
    assert madd > 20 * np.median(kth)                                     # the window swallows the k-th distance


def test_pivot_starvation_puts_every_pivot_on_one_chromosome():
    for zero in (0, 150):
        case = pivot_starved(zero_rows=zero)
        X, bins = case["X"], case["bins"]
        n32 = norms(X).astype(np.float32)                                 # K4h hands the pivot select fp32 norms
        piv = np.lexsort((np.arange(len(n32)), n32))[:TC_PIVOTS]
        c = chrom_of(bins)[piv]
        if zero:
            assert (c == len(bins) - 1).sum() == zero and set(c) == {0, len(bins) - 1}
            assert (X[-zero:] == 1.0).all()
        else:
            assert (c == 0).all()


@pytest.mark.parametrize("rank", [3, 5])
def test_low_rank_crowds_the_window(rank):
    case = low_rank(rank)
    X, bins, k = case["X"], case["bins"], case["k"]
    sv = np.linalg.svd(X - 1.0, compute_uv=False)
    assert sv[rank] < 1e-2 * sv[rank - 1]
    nrm = norms(X)
    e = eps16(X.shape[1])
    crowd = []
    for t in _sample_targets(case, 20, seed=2):
        cand, d = exact_row(X, bins, t)
        dk = np.sort(d)[k - 1]
        crowd.append(np.sum(np.abs(d - dk) <= e * (nrm[t] + nrm[cand])))
    assert np.median(crowd) >= 2                                          # the k-th distance is a near tie


@pytest.mark.parametrize("S", [1, 8])
def test_range_boundary_distances_straddle_1e10(S):
    case = range_boundary(S)
    X, bins = case["X"], case["bins"]
    lo, hi = np.nextafter(1e10, 0.0), np.nextafter(1e10, np.inf)
    if S == 1:
        lo, hi = np.nextafter(lo, 0.0), np.nextafter(hi, np.inf)
    nt = bins[0]
    for t in range(nt):
        rows = nt + case["steps"] * t + np.arange(3)
        d = wc_oracle.squared_distances_seq(X[rows], X[t])
        assert d[0] == 1e10 and d[1] == lo and d[2] == hi
    sp = X[-10:, 0]
    assert np.signbit(sp[0]) and sp[0] == 0.0 and sp[1] == 1.0 and np.isnan(sp[2]) and sp[3] == np.inf and sp[4] == -np.inf
    assert np.abs(X[nt:nt + bins[1]] - 1.0).max() > FP16_LIMIT                 # every filter option runs the fp64 filter


def test_pca_matrix_with_sparse_bins_widens_the_fp16_window():
    """Point of the sparse PCA family (250 kb, S = 200): the largest |x - 1| is ~1e2, n_max / 2 stays inside fp16's
    range, and filt_madd is ~2 orders of magnitude above a typical row's k-th distance."""
    from wisecondor_b200 import synth as _s
    counts, bins = pca_counts(250000, 200, sparse=True)
    samples = [_s.counts_to_sample_dict(counts[i], bins, 250000) for i in range(counts.shape[0])]
    masked, chrom_bins, mask = wc_oracle.to_numpy_array(samples)
    corrected, comps, mean = wc_oracle.train_pca(masked)
    sizes = masked_sizes(chrom_bins, mask)
    nrm = norms(corrected)
    assert 50 < np.abs(corrected - 1.0).max() < FP16_LIMIT and nrm.max() / 2 < FP16_LIMIT
    kth = []
    for t in np.random.default_rng(4).choice(corrected.shape[0], 10, replace=False):
        cand, d = exact_row(corrected, sizes, t)
        kth.append(np.sort(d)[K - 1])
    assert filt_madd(200, nrm.max()) > 20 * np.median(kth)
    counts0, _ = pca_counts(250000, 200, sparse=False)
    assert (counts0 != counts).sum() == 20
