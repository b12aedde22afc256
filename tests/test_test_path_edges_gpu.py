"""Adversarial parity of the test path's device kernels against plain high-precision references.

K9 (segmentation): exact ties across positions and lengths, repeated blocks, mirror pairs, thresholds equal to a run's
value, large dynamic range (the all-rows fallback), chained spikes (more than 128 pending ranges, more than 256 calls),
z near the top of the fp32 and fp64 ranges and full chromosome sizes, against wc_oracle.segment_region (n <= 400) or
wc_oracle.segment_region_exact: calls exact, call z and chromosome-wide z bit-identical.

K8 (z-scores): every sample of batches of 31 to 100 samples, refsize 20 to 512, with NaN / +inf / negative / +-0 test
values in heavily used reference bins and both later-pass kernels (dirty-pair list and full pass) exercised, against
wc_oracle.repeat_test: z, r, refsizes bit-identical (NaN-equal), sigma average equal."""
import time

import numpy as np
import pytest

import c_oracle
import wc_oracle
from test_segment_exact_oracle import adversarial_regions, chained_spikes, threshold_at_call, _square_ties
from wisecondor_b200 import synth

pytestmark = pytest.mark.gpu


# ---- K9 ------------------------------------------------------------------------------------------------------------
def _segment(z, thr, min_search=3, r=None, t=0.0):
    """One region as one sample with a single chromosome: (chromosome-wide z, [(z, (x, y)), ...])."""
    from wisecondor_b200 import wisetools
    n = len(z)
    cwz, cleaned, calls = wisetools.segmentChromosomes(z[None, :], np.full((1, n), 100), [n], [1], 25, thr, min_search,
                                                       resultsR=None if r is None else r[None, :], mineffectsize=t)
    assert int(cleaned[0, 0]) == n
    segs = [(float(c["z"]), (int(c["x"]), int(c["y"]))) for c in calls]
    assert all(0 <= x <= y < n for _, (x, y) in segs)
    return float(cwz[0, 0]), segs


def _oracle(z, thr, min_search=3):
    if len(z) <= 400:
        with np.errstate(over="ignore"):
            return wc_oracle.segment_region(z, thr, min_search)
    return wc_oracle.segment_region_exact(z, thr, min_search)


def _assert_same(got, want, what):
    assert got[0] == want[0], "%s: chromosome-wide z %r vs %r" % (what, got[0], want[0])
    assert [s[1] for s in got[1]] == [s[1] for s in want[1]], "%s: calls %s vs %s" % (what, got[1][:8], want[1][:8])
    assert [s[0] for s in got[1]] == [float(s[0]) for s in want[1]], "%s: call z" % what


SMALL = [(name, z, thr) for n, seed in [(40, 11), (131, 12), (300, 13)] for name, z, thr in adversarial_regions(n, seed)]


@pytest.mark.parametrize("i", range(len(SMALL)), ids=["%s-%d" % (c[0], len(c[1])) for c in SMALL])
def test_k9_adversarial_families_vs_full_triangle(i):
    name, z, thr = SMALL[i]
    _assert_same(_segment(z, thr), _oracle(z, thr), name)


def test_k9_threshold_equal_to_a_run_value():
    """abs(champVal) < threshold is False at equality: the run is called at its own exact value and at the next double
    below it, not at the next double above."""
    rng = np.random.default_rng(17)
    regions = [rng.integers(-3, 4, size=90).astype(float), rng.integers(-12, 13, size=150) / 4.0, _square_ties(rng, 70),
               rng.normal(0, 1, size=200)]
    for k, z in enumerate(regions):
        t_eq, t_below, t_above = threshold_at_call(z)
        for t in (t_eq, t_below, t_above):
            got, want = _segment(z, t), _oracle(z, t)
            _assert_same(got, want, "region %d thr %r" % (k, t))
        assert len(_segment(z, t_eq)[1]) >= 1


@pytest.mark.parametrize("family", ["int", "dyadic", "square_ties", "spike1e6", "spike1e12", "spike1e30", "fp32_1e37"])
def test_k9_min_effect_on_ties_and_dynamic_range(family):
    """fillTriMin's median filter with ratios rounded to 2 decimals (exact ties at the effect boundary)."""
    rng = np.random.default_rng(23)
    for n, seed in [(60, 31), (170, 32)]:
        z, thr = {name: (zz, tt) for name, zz, tt in adversarial_regions(n, seed)}[family]
        r = np.round(1.0 + rng.normal(0, 0.05, size=n) + 0.02 * np.sign(z), 2)
        t = 0.05
        got = _segment(z, thr, r=r, t=t)
        with np.errstate(over="ignore"):
            want = wc_oracle.segment_region(z, thr, 3, r, t)
        _assert_same(got, want, "%s n=%d" % (family, n))


@pytest.mark.parametrize("family", ["spike1e6", "spike1e12", "spike1e30", "tiny", "offset", "fp32_1e37",
                                    "fp32_1e37_wide", "fp32_2e38", "fp64_1e300"])
def test_k9_dynamic_range_2000_bins(family):
    """After a huge spike is called the noise ranges' error window (scaled by sum |z| of the chromosome) admits every
    run: the all-rows path re-scores them all exactly.  Its time is printed, not asserted."""
    z, thr = {name: (zz, tt) for name, zz, tt in adversarial_regions(2000, 41)}[family]
    t0 = time.perf_counter()
    got = _segment(z, thr)
    ms = (time.perf_counter() - t0) * 1e3
    from wisecondor_b200 import device
    print("K9 %s n=2000: %.1f ms wall, %.2f ms segmentation kernel, %d calls"
          % (family, ms, device.last_test_stats()["segment_ms"], len(got[1])))
    _assert_same(got, wc_oracle.segment_region_exact(z, thr, 3), family)


@pytest.mark.parametrize("k", [140, 400])
def test_k9_chained_spikes_more_pending_ranges_than_128(k):
    """k spikes 5 bins apart: up to k ranges are pending at once (the stack holds n / (min_search + 1) + 1)."""
    z = chained_spikes(k)
    got = _segment(z, 5.0)
    want = wc_oracle.segment_region_exact(z, 5.0, 3)
    assert len(want[1]) == k
    _assert_same(got, want, "k=%d" % k)


def test_k9_more_calls_than_max_calls_in_a_batch():
    """One sample with 400 calls (device.segment_batch retries with a larger max_calls) next to ordinary samples, with
    min_search 0 as well."""
    import torch
    from wisecondor_b200 import device
    rng = np.random.default_rng(5)
    n = 2005
    for ms in (3, 0):
        Z = rng.normal(0, 1, size=(3, n))
        Z[1] = chained_spikes(400, seed=2)
        Z[2, 100:140] += 2.0
        zd = torch.from_numpy(Z).cuda()
        sizes = torch.full((3, n), 100, dtype=torch.int32, device="cuda")
        cwz, cleaned, calls = device.segment_batch(zd, sizes, [n], [0], 25, 5.0, ms)
        assert (calls["sample"] == 1).sum() >= 400
        for b in range(3):
            want = wc_oracle.segment_region_exact(Z[b], 5.0, ms)
            mine = calls[calls["sample"] == b]
            got = (float(cwz[b, 0].item()), [(float(c["z"]), (int(c["x"]), int(c["y"]))) for c in mine])
            _assert_same(got, want, "sample %d min_search %d" % (b, ms))


def test_k9_fp64_overflow_is_a_clean_error():
    """sum |z| at or beyond 2^1023 could overflow numpy's run sums: the whole batch is refused with WC_ERR_ARG and a
    message saying so - never a call outside [0, n).  Just below that bound the result is the reference's, bit for
    bit."""
    from wisecondor_b200 import _cabi
    rng = np.random.default_rng(3)
    n = 120
    for pattern in ([1e308, 1e308], [1.7e308, -1.7e308, 1.7e308], [9e307] * 4):
        z = rng.normal(0, 1, size=n)
        z[50:50 + len(pattern)] = pattern
        with pytest.raises(_cabi.WisecondorError, match="2\\^1023"):
            _segment(z, 4.0)
    z = rng.normal(0, 1, size=n)
    z[30] = 8.9e307                                   # sum |z| < 2^1023 = 8.988e307
    z[80:90] += 3.0
    _assert_same(_segment(z, 4.0), _oracle(z, 4.0), "below 2^1023")
    z[31] = -8.9e307                                  # the two cancel: every run sum stays finite, sum |z| does not
    with pytest.raises(_cabi.WisecondorError, match="2\\^1023"):
        _segment(z, 4.0)


def _chromosome_batch(bins, B, seed):
    rng = np.random.default_rng(seed)
    n = int(sum(bins))
    Z = rng.normal(0, 1, size=(B, n))
    for b in range(B):
        for _ in range(6):
            a = int(rng.integers(0, n - 400))
            Z[b, a:a + int(rng.integers(5, 400))] += rng.choice([-1.2, 0.8, 2.5])
    sizes = rng.integers(20, 120, size=(B, n)).astype(np.int32)
    return Z, sizes


def _check_batch(Z, sizes, bins, chroms, thr, cwz, calls, samples):
    starts = np.concatenate(([0], np.cumsum(bins)))
    for b in samples:
        for slot, c in enumerate(chroms):
            keep = sizes[b, starts[c]:starts[c + 1]] >= 25
            zc = Z[b, starts[c]:starts[c + 1]][keep]
            want = wc_oracle.segment_region_exact(zc, thr, 3)
            mine = calls[(calls["sample"] == b) & (calls["chrom"] == slot)]
            got = (float(cwz[b, slot]), [(float(m["z"]), (int(m["x"]), int(m["y"]))) for m in mine])
            _assert_same(got, want, "sample %d chromosome %d" % (b, c))


def test_k9_full_size_chromosomes():
    """A 50 kb-shaped batch (chr1 about 5 000 kept bins: prefix sums, side arrays and range stack in shared memory), a
    10 kb-sized chromosome (25 000 bins: prefix sums and side arrays fill 200 KB of shared memory, the range stack moves
    to global scratch) and a 30 000-bin one (the side arrays move to global scratch, the stack sits after the prefix
    sums in shared memory)."""
    import torch
    from wisecondor_b200 import device
    bins = [int(v) for v in synth.chrom_bins(50000)]
    Z, sizes = _chromosome_batch(bins, 3, 1)
    chroms = list(range(22))
    cwz, cleaned, calls = device.segment_batch(torch.from_numpy(Z).cuda(), torch.from_numpy(sizes).cuda(), bins, chroms,
                                               25, 4.5, 3)
    assert len(calls) >= 3
    _check_batch(Z, sizes, bins, chroms, 4.5, cwz.cpu().numpy(), calls, [0, 2])

    # (no huge spike here: the ranges beside it would take the O(m^3) all-rows path, minutes at this size)
    for n in (25000, 30000):
        Z, sizes = _chromosome_batch([n], 2, 2)
        t0 = time.perf_counter()
        cwz, cleaned, calls = device.segment_batch(torch.from_numpy(Z).cuda(), torch.from_numpy(sizes).cuda(),
                                                   [n], [0], 25, 5.0, 3)
        print("K9 %d bins, 2 samples: %.1f ms, %d calls" % (n, (time.perf_counter() - t0) * 1e3, len(calls)))
        assert len(calls) >= 2
        _check_batch(Z, sizes, [n], [0], 5.0, cwz.cpu().numpy(), calls, [0, 1])


# ---- K8 ------------------------------------------------------------------------------------------------------------
def _global_table(idx, dst, bins, cutoff):
    """Usable reference bins of every bin in global coordinates (idx[distances < cutoff] out of the other-chromosome
    concatenation, wisetools.py:420-424) as a dense bins x bins usage matrix."""
    n = int(sum(bins))
    use = np.zeros((n, n), dtype=bool)
    starts = np.concatenate(([0], np.cumsum(bins)))
    for c in range(len(bins)):
        cs, ce = starts[c], starts[c + 1]
        for i in range(cs, ce):
            j = idx[i][dst[i] < cutoff]
            use[i, j + np.where(j >= cs, ce - cs, 0)] = True
    return use


def _passes(test, copy0, idx, dst, bins, sums, cutoff, thr, repeats):
    """repeatTest from a given working copy: every pass's (z, r, sizes, sd avg) and the copy before each pass."""
    copy = np.copy(copy0)
    outs, copies = [], []
    for _ in range(repeats):
        copies.append(np.copy(copy))
        out = wc_oracle.try_sample(test, copy, idx, dst, bins, sums, cutoff)
        outs.append(out)
        with np.errstate(invalid="ignore"):
            copy[np.abs(out[0]) >= thr] = -1
    return outs, copies


@pytest.mark.parametrize("B,k,regime", [(31, 20, "few"), (33, 100, "many"), (64, 129, "few"), (65, 512, "many"),
                                        (100, 100, "few"), (100, 20, "many")])
def test_k8_every_sample_special_values_and_both_later_pass_kernels(B, k, regime):
    """Every sample of the batch against the oracle.  NaN, +inf, -1, -0.5, -0.0 and 0.0 test values sit in the bins
    most used as reference bins (the reverse index); half the samples also start from a pre-marked copy (copy_init).
    The later passes recompute either the listed dirty pairs or, past N*B/8 pairs, every pair: the test models the
    dirty set from the oracle's marks and the usage table and checks the device's per-pass counts against it."""
    import torch
    from wisecondor_b200 import device
    bins = [int(b) for b in np.maximum(3, np.array(synth.chrom_bins(250000)) // 12)]
    n = sum(bins)
    sums = list(np.cumsum(bins))
    X = synth.corrected_like(bins, 16, seed=B + k)
    idx, dst = c_oracle.get_reference_rows(X, bins, 0, n, k)
    cutoff = wc_oracle.get_optimal_cutoff(dst, 3)
    use = _global_table(idx, dst, bins, cutoff)
    hot = np.argsort(-use.sum(axis=0), kind="stable")[:24]          # the most used reference bins
    rng = np.random.default_rng(B * 1000 + k)
    tests = 1.0 + rng.normal(0, 0.03, size=(B, n))
    # "few": threshold 5, mild aberrations and the special values in two samples only, so that the marks dirty fewer
    # than N*B/8 pairs; "many": threshold 1.2, strong aberrations and special values in every sample
    few = regime == "few"
    thr = 5.0 if few else 1.2
    specials = [np.nan, np.inf, -1.0, -0.5, -0.0, 0.0]
    for b in range(B):
        a = int(rng.integers(0, n - 40))
        tests[b, a:a + int(rng.integers(3, 40))] *= rng.choice([0.97, 1.03] if few else [0.8, 1.2])
        if not few or b in (0, B - 1):
            for j, v in enumerate(specials):
                tests[b, hot[(b + 4 * j) % len(hot)]] = v
    copy0 = np.copy(tests)
    for b in range(0, B, 2):                                         # arbitrary pre-marks, some on the special bins
        copy0[b, rng.random(n) < 0.05] = -1.0
        copy0[b, hot[b % len(hot)]] = -1.0
    repeats = 4
    ldb = device.pad32(B)
    T = torch.ones((n, ldb), dtype=torch.float64, device="cuda")
    C = torch.ones((n, ldb), dtype=torch.float64, device="cuda")
    T[:, :B] = torch.from_numpy(np.ascontiguousarray(tests.T)).cuda()
    C[:, :B] = torch.from_numpy(np.ascontiguousarray(copy0.T)).cuda()
    table = device.ReferenceTable(idx, dst, bins, cutoff)
    z, r, sizes, asdef = device.zscore_batch(T, B, table, thr, repeats, copy_init=C)
    pairs = device.last_test_stats()["zscore_pairs_per_pass"]
    z, r, sizes, asdef = z.cpu().numpy(), r.cpu().numpy(), sizes.cpu().numpy(), asdef.cpu().numpy()

    newly = np.zeros((repeats, n, B), dtype=bool)                    # newly marked (bin, sample) before pass p
    for b in range(B):
        outs, copies = _passes(tests[b], copy0[b], idx, dst, bins, sums, cutoff, thr, repeats)
        want = outs[-1]
        assert np.array_equal(z[b], want[0], equal_nan=True), "sample %d z" % b
        assert np.array_equal(r[b], want[1], equal_nan=True), "sample %d r" % b
        assert np.array_equal(sizes[b], want[2]), "sample %d refsizes" % b
        assert asdef[b] == want[3] or (np.isnan(asdef[b]) and np.isnan(want[3])), "sample %d sigma" % b
        for p in range(1, repeats):
            newly[p, :, b] = (copies[p] == -1.0) & (copies[p - 1] != -1.0)
    limit = n * B // 8
    kinds = []
    for p in range(1, repeats):
        dirty = int((use.astype(np.int32) @ newly[p].astype(np.int32) > 0).sum())
        assert pairs[p] == (dirty if dirty <= limit else n * B), "pass %d: %d dirty pairs, device %d" % (p, dirty, pairs[p])
        kinds.append("pairs" if dirty <= limit else "full")
    if regime == "few":
        assert "pairs" in kinds and any(pairs[p] > 0 for p in range(1, repeats))
    else:
        assert "full" in kinds


# ---- full shape -------------------------------------------------------------------------------------------------------
def test_full_shape_two_samples_vs_oracles():
    """test_full_size_properties_50kb's workload (57 633 bins, refsize 100, 48 samples): two samples' z, r, refsizes and
    sigma average against wc_oracle.repeat_test and their calls and chromosome-wide z against segment_region_exact."""
    import torch
    from wisecondor_b200 import device
    bins = synth.chrom_bins(50000)
    n = int(sum(bins))
    sums = list(np.cumsum(bins))
    X = torch.from_numpy(synth.corrected_like(bins, 64, seed=4)).cuda()
    idx, dist = device.newref_topk(X, bins, 0, n, 100)
    idx_h, dist_h = idx.cpu().numpy(), dist.cpu().numpy()
    cutoff = wc_oracle.get_optimal_cutoff(dist_h, 3)
    table = device.ReferenceTable(idx_h, dist_h, bins, cutoff)
    rng = np.random.default_rng(2)
    B = 48
    host = 1.0 + rng.normal(0, 0.03, size=(B, n))
    for b in range(B):
        a = int(rng.integers(0, n - 500))
        host[b, a:a + int(rng.integers(20, 400))] *= rng.choice([0.85, 1.15])
    thr = 5.4
    T = torch.ones((n, device.pad32(B)), dtype=torch.float64, device="cuda")
    T[:, :B] = torch.from_numpy(np.ascontiguousarray(host.T)).cuda()
    z, r, sizes, asdef = device.zscore_batch(T, B, table, thr, 5)
    cwz, cleaned, calls = device.segment_batch(z, sizes, bins, list(range(22)), 25, thr, 3)
    z, r, sizes, asdef, cwz = z.cpu().numpy(), r.cpu().numpy(), sizes.cpu().numpy(), asdef.cpu().numpy(), cwz.cpu().numpy()
    for b in (0, B - 1):
        want = wc_oracle.repeat_test(host[b], idx_h, dist_h, bins, sums, cutoff, thr, 5)
        assert np.array_equal(z[b], want[0], equal_nan=True) and np.array_equal(r[b], want[1], equal_nan=True)
        assert np.array_equal(sizes[b], want[2]) and asdef[b] == want[3]
    _check_batch(z, sizes, bins, list(range(22)), thr, cwz, calls, [0, B - 1])
