"""GPU parity of the reference-bin search on adversarial inputs (tests/test_search_adversarial_inputs.py) and at the
parameter edges of its kernels: every result must equal the C oracle's - identical indexes, bit-identical distances -
under every filter (k5_f16 = 2 tcgen05, 1 mma.sync, 0 fp64) and both K6 selects (k6_select = 1 histogram, 0 bisection).
Also: the fp16 filter's computed distances against the a-priori bound on those inputs, and the device PCA at production
sample counts (S = 200, 600, 2000: off-diagonal Gram tiles, numpy's pairwise mean above one 128-element block), whose
corrected matrix then feeds the search.  Each search prints its counters (`EDGE-STATS ...`, visible with -s)."""
import ctypes
import hashlib
import os

import numpy as np
import pytest

import c_oracle
import test_search_adversarial_inputs as A
import wc_oracle
from wisecondor_b200 import _cabi, synth

pytestmark = [pytest.mark.gpu]

DEFAULT_FILTER = int(os.environ.get("WC_K5_F16", "2"))        # the context's defaults
DEFAULT_SELECT = 1
_ORACLE = {}


def _setopt(key, value):
    _cabi.check(_cabi.lib().wc_set_option(_cabi.context(0).handle, key.encode(), float(value)))


@pytest.fixture(params=[(2, 1), (2, 0), (1, 1), (1, 0), (0, 1), (0, 0)],
                ids=["tc-hist", "tc-bisect", "mma-hist", "mma-bisect", "fp64-hist", "fp64-bisect"])
def opts(request):
    f16, select = request.param
    _setopt("k5_f16", f16)
    _setopt("k6_select", select)
    yield dict(k5_f16=f16, k6_select=select)
    _setopt("k5_f16", DEFAULT_FILTER)
    _setopt("k6_select", DEFAULT_SELECT)


def _search(X, bins, r0, r1, k):
    from wisecondor_b200 import device
    idx, dist = device.newref_topk_host(X, bins, r0, r1, k)
    return idx, dist, device.last_search_stats(0)


def _report(name, st, **extra):
    keys = ("filter", "exhaustive_rows", "k6_live_max", "k6_shortlisted", "pivots", "dist_topk_ms", "finalize_ms",
            "exhaustive_ms")
    print("EDGE-STATS %s %s %s" % (name, " ".join("%s=%s" % kv for kv in extra.items()),
                                   " ".join("%s=%s" % (key, round(st[key], 3) if isinstance(st[key], float) else st[key])
                                            for key in keys)))


def _assert_same(idx, dist, oidx, odist, what=""):
    assert idx.shape == oidx.shape and dist.shape == odist.shape
    bad = np.flatnonzero((idx != oidx).any(axis=1) | ~(dist.view(np.int64) == odist.view(np.int64)).all(axis=1))
    assert bad.size == 0, "%s: %d rows differ, first %s: %s / %s vs %s / %s" % (
        what, bad.size, bad[:8], idx[bad[0]][:8], dist[bad[0]][:4], oidx[bad[0]][:8], odist[bad[0]][:4])


def _oracle(case):
    """The C oracle on every row, computed once per input (cases are regenerated for every option set)."""
    key = (case["k"], tuple(case["bins"]), hashlib.sha1(case["X"].tobytes()).hexdigest())
    if key not in _ORACLE:
        _ORACLE[key] = c_oracle.get_reference_rows(case["X"], case["bins"], 0, case["X"].shape[0], case["k"])
    return _ORACLE[key]


def _expected_filter(case, mode):
    if case["name"].startswith("range_boundary") or case["name"] == "fp16_edge_value":
        return 0                                         # |x - 1| > 60000: every option runs the fp64 filter
    if case["name"] == "fp16_edge_above" and mode == 2:
        return 0                                         # n / 2 > 60000: the tcgen05 path's folded norms leave fp16's range
    return mode


def _check_all_rows(case, tag):
    """Whole-matrix call (symmetric search where N allows) and a row-range call (plain search), both against the oracle."""
    X, bins, k = case["X"], case["bins"], case["k"]
    n = X.shape[0]
    oidx, odist = _oracle(case)
    idx, dist, st = _search(X, bins, 0, n, k)
    _assert_same(idx, dist, oidx, odist, case["name"] + " whole")
    _report(case["name"], st, opts=tag, call="whole")
    r0, r1 = n // 3 + 7, min(n, n // 3 + 7 + 700)
    idx, dist, st2 = _search(X, bins, r0, r1, k)
    _assert_same(idx, dist, oidx[r0:r1], odist[r0:r1], case["name"] + " rows")
    return st


# ---------------------------------------------------------------------------------------------------------------------
# every family under every filter and select
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family", list(A.FAMILIES))
def test_family_equals_oracle(family, opts):
    case = A.FAMILIES[family]()
    st = _check_all_rows(case, "f%d-s%d" % (opts["k5_f16"], opts["k6_select"]))
    assert st["filter"] == _expected_filter(case, opts["k5_f16"])
    if family in A.NO_FALLBACK:
        assert st["exhaustive_rows"] == 0


@pytest.mark.parametrize("family", ["near_tie_M200_d1e-07", "near_tie_M101_d1e-03", "tie_shell", "sigma_mix",
                                    "sparse_rows", "pivot_starved", "pivot_starved_zero", "low_rank_3"])
@pytest.mark.parametrize("world", [2, 3])
def test_family_sharded_equals_oracle(family, world):
    """The block pairs of the symmetric search divided over `world` ranks (emulated on one GPU)."""
    from test_search_shard_gpu import _emulated_ranks
    case = A.FAMILIES[family]()
    oidx, odist = _oracle(case)
    idx, dist, stats = _emulated_ranks(case["X"], case["bins"], case["k"], world)
    _assert_same(idx, dist, oidx, odist, "%s W=%d" % (family, world))


# ---------------------------------------------------------------------------------------------------------------------
# parameter edges (default options), all rows against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def _edge_cases(S=64, k=A.K, bins=None):
    bins = list(A.MID_BINS if bins is None else bins)
    chrom = int(np.argsort(bins)[-2]) if len(bins) > 1 else 0          # the cluster on the second largest chromosome
    M = max(2, min(2 * k, bins[chrom]))
    return [A.plain(S=S, k=k, bins=bins, seed=S + k),
            A.near_tie(M, 1e-7, S=S, k=k, bins=bins, chrom=chrom, seed=S + k)]


@pytest.mark.parametrize("S", [59, 60, 61, 63, 64, 65, 99, 100, 101, 124, 125, 127, 128, 129])
def test_sample_count_edges(S):
    """ldh = ceil((S + 4) / 64) * 64, K6c's 100-sample chunk, S % 4 (vector loads in K6), odd S (the fused K6)."""
    for case in _edge_cases(S=S):
        _check_all_rows(case, "S%d" % S)


@pytest.mark.parametrize("k", [1, 31, 32, 33, 96, 97, 128, 129, 255, 256, 257, 384])
def test_refsize_edges(k):
    """shortcap 256 / 512 (96 / 97 under the fp16 filter), cap 512 / 1024 and pivots on / off (128 / 129), bitonic sizes."""
    for case in _edge_cases(k=k):
        _check_all_rows(case, "k%d" % k)


def _scaled_bins(n, nchrom=22):
    base = np.array(A.MID_BINS[:nchrom], dtype=float)
    bins = np.maximum(1, np.floor(base / base.sum() * n)).astype(int)
    bins[0] += n - bins.sum()
    return [int(b) for b in bins]


LAYOUTS = {
    "N2944_plain": _scaled_bins(2944),                       # 23 row blocks: the plain search
    "N2945_sym": _scaled_bins(2945),                         # 24 row blocks: the symmetric search
    "N2047_nopivots": _scaled_bins(2047),                    # 4 * TC_PIVOTS > N: no pivot pass
    "N2048_pivots": _scaled_bins(2048),
    "N3001": _scaled_bins(3001),                             # N not a multiple of 128
    "block_edges": [128 * m for m in (3, 2, 4, 1, 5, 2, 3, 2, 1, 1, 2, 4)],      # every chromosome ends on a block edge
    "one_bin_chroms": [1] * 150 + [1400, 1200, 700] + [1] * 50,
    "one_chrom_90pct": [3456, 130, 120, 80, 54],
}


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_layout_edges(layout):
    for case in _edge_cases(bins=LAYOUTS[layout]):
        _check_all_rows(case, layout)


# ---------------------------------------------------------------------------------------------------------------------
# the fp16 filter's distances against the bound its margins are built on
# ---------------------------------------------------------------------------------------------------------------------
QUARTER = [int(b) for b in np.maximum(1, np.array(synth.chrom_bins(250000)) // 4)]


def _bound_cases():
    yield A.near_tie(200, 1e-5, bins=QUARTER)
    yield A.sigma_mix()
    yield A.low_rank(3)
    yield A.sparse_rows()
    for S in (60, 61, 63, 125):
        yield A.plain(S=S, bins=QUARTER)
        yield A.near_tie(200, 1e-3, S=S, bins=QUARTER)


def test_tc_filter_distances_stay_inside_the_bound_on_adversarial_inputs():
    """Every filter distance the tcgen05 kernel computes (wc_debug_filter_scores) lies within eps16 (n_i + n_j) plus the
    subnormal term of the fp64 distance - the premise of the search's exactness, tested directly."""
    import torch
    from wisecondor_b200 import device
    L = _cabi.lib()
    ctx = _cabi.context(0)
    for case in _bound_cases():
        X, bins = case["X"], case["bins"]
        n, S = X.shape
        out = torch.full((n, n), float("nan"), dtype=torch.float32, device="cuda:0")
        _setopt("k5_f16", 2)
        _setopt("k5_sym", 0)
        _cabi.check(L.wc_debug_filter_scores(ctx.handle, ctypes.c_void_p(out.data_ptr()), n))
        try:
            device.newref_topk(torch.as_tensor(X, device="cuda:0"), bins, 0, n, 50)
            torch.cuda.synchronize()
        finally:
            _cabi.check(L.wc_debug_filter_scores(ctx.handle, None, 0))
            _setopt("k5_f16", DEFAULT_FILTER)
            _setopt("k5_sym", 8)
        got = out.cpu().numpy().astype(np.float64)
        del out
        xc = X - 1.0
        nrm = (xc * xc).sum(axis=1)
        exact = nrm[:, None] + nrm[None, :] - 2.0 * (xc @ xc.T)
        computed = ~np.isnan(got)
        chrom = A.chrom_of(bins)
        other = chrom[:, None] != chrom[None, :]
        assert computed[other].all(), "%s: tiles missing" % case["name"]
        bound = A.eps16(S) * (nrm[:, None] + nrm[None, :]) + A.filter_sub(S, nrm.max())
        ratio = (np.abs(got - exact)[computed] / bound[computed]).max()
        print("EDGE-STATS bound %s S=%d max |d~ - d| / bound = %.3g" % (case["name"], S, ratio))
        assert ratio <= 1.0, case["name"]


# ---------------------------------------------------------------------------------------------------------------------
# device PCA at production sample counts, and the search on its output
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("binsize,S,sparse", [(250000, 200, False), (250000, 200, True), (50000, 600, False),
                                              (50000, 600, True), (250000, 2000, False)],
                         ids=["250kb-S200", "250kb-S200-sparse", "50kb-S600", "50kb-S600-sparse", "250kb-S2000"])
def test_device_pca_then_search(binsize, S, sparse):
    from wisecondor_b200 import wisetools
    counts, bins = A.pca_counts(binsize, S, sparse)
    samples = [synth.counts_to_sample_dict(counts[i], bins, binsize) for i in range(S)]
    masked, chrom_bins, mask = wisetools.toNumpyArray(samples)
    corrected, pca = wisetools.trainPCA(masked)
    omasked, ochrom_bins, omask = wc_oracle.to_numpy_array(samples)
    assert np.array_equal(mask, omask) and np.array_equal(masked, omasked)
    ocorr, ocomps, omean = wc_oracle.train_pca(omasked)
    assert np.array_equal(pca.mean_, omean)                                   # bit for bit: numpy's pairwise order
    rel = np.abs(corrected - ocorr) / np.maximum(np.abs(ocorr), 1e-300)
    assert rel.max() <= 1e-9, "corrected: max rel %g" % rel.max()
    for j in range(ocomps.shape[0]):
        sign = 1.0 if np.dot(pca.components_[j], ocomps[j]) >= 0 else -1.0
        assert np.abs(sign * pca.components_[j] - ocomps[j]).max() <= 1e-9 * np.abs(ocomps[j]).max(), "component %d" % j
    # the device's corrected matrix is the input of both searches: the comparison stays bit-exact
    sizes = A.masked_sizes(chrom_bins, mask)
    n = corrected.shape[0]
    idx, dist, st = _search(corrected, sizes, 0, n, A.K)
    _report("pca_%dkb_S%d%s" % (binsize // 1000, S, "_sparse" if sparse else ""), st, N=n)
    sums = np.cumsum(sizes)
    for r0 in sorted({0, int(sums[0]) - 16, int(sums[6]) - 16, n // 2, n - 32}):
        oidx, odist = c_oracle.get_reference_rows(corrected, sizes, r0, r0 + 32, A.K)
        _assert_same(idx[r0:r0 + 32], dist[r0:r0 + 32], oidx, odist, "rows %d.." % r0)
    assert (np.diff(dist, axis=1) >= 0).all()
    if not sparse:
        assert st["exhaustive_rows"] == 0
