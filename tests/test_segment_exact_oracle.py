"""CPU pin of wc_oracle.segment_region_exact against segment_region (the full triangle in the reference's own order) on
small regions of every adversarial family the GPU segmentation tests use: exact ties across positions and lengths,
repeated blocks, mirror pairs, thresholds equal to a run's value, large dynamic range, chained spikes and z near the
top of the fp32 and fp64 ranges.  segment_region_exact is the oracle of those tests at chromosome sizes where
segment_region is out of reach; it must return the same calls and values bit for bit wherever both run."""
import numpy as np
import pytest

import wc_oracle


def _square_ties(rng, n):
    """Runs of exactly equal value 2 at lengths 1, 4 and 16 (2/1 = 4/2 = 8/4) and their negatives, in random order and
    apart by -3 / +3 padding so that joined runs are smaller: the row-major first occurrence and the +/- rule decide."""
    blocks = [[2.0], [1.0] * 4, [0.5] * 16, [-2.0], [-1.0] * 4, [-0.5] * 16]
    order = rng.permutation(len(blocks))
    z = []
    for i in order:
        z.extend(blocks[i])
        z.extend([-3.0 if blocks[i][0] > 0 else 3.0] * 2)
    z = np.array(z)
    return np.concatenate((z, rng.integers(-1, 2, size=max(0, n - len(z))).astype(float)))


def _repeated(rng, n):
    pat = rng.integers(-3, 4, size=int(rng.integers(3, 9))).astype(float)
    pat[0] = 4.0
    z = rng.integers(-1, 2, size=n).astype(float)
    for off in range(2, n - len(pat), max(len(pat) + 3, n // 5)):
        z[off:off + len(pat)] = pat
    return z


def _mirror(rng, n):
    z = np.round(rng.normal(0, 0.5, size=n) * 4) / 4
    w = int(rng.integers(2, 9))
    a = float(rng.integers(2, 6))
    for off in range(3, n - 2 * w, max(2 * w + 5, n // 3)):
        if rng.random() < 0.5:
            z[off:off + w], z[off + w:off + 2 * w] = -a, a          # the negative first: the positive still wins
        else:
            z[off:off + w], z[off + w:off + 2 * w] = a, -a
    return z


def _spike(rng, n, height):
    """One huge bin among N(0, 1) noise, and a +-2.5 stretch that the recursion calls next to it in the noise."""
    z = rng.normal(0, 1, size=n)
    s = int(rng.integers(0, n))
    b = (s + n // 2) % n
    b = min(b, n - 12)
    z[b:b + 12] += 2.5 * rng.choice([-1.0, 1.0])
    z[s] = height * rng.choice([-1.0, 1.0])
    return z


def chained_spikes(k, seed=0):
    """k spikes at bins 5j + 2 of magnitude 10 + 0.1 j with alternating sign over N(0, 0.1) noise (5k + 5 bins):
    with threshold 5 and min_search 3 every spike is called and up to k ranges are pending at once."""
    rng = np.random.default_rng(seed)
    z = rng.normal(0, 0.1, size=5 * k + 5)
    for j in range(k):
        z[5 * j + 2] = (10.0 + 0.1 * j) * (1 if j % 2 == 0 else -1)
    return z


def adversarial_regions(n, seed):
    """(family, z, threshold) triples of length about n."""
    rng = np.random.default_rng(seed)
    out = [
        ("int", rng.integers(-3, 4, size=n).astype(float), 3.0),
        ("dyadic", rng.integers(-12, 13, size=n) / 4.0, 2.5),
        ("square_ties", _square_ties(rng, n), 1.5),
        ("repeated", _repeated(rng, n), 3.0),
        ("mirror", _mirror(rng, n), 2.0),
        ("spike1e6", _spike(rng, n, 1e6), 4.0),
        ("spike1e12", _spike(rng, n, 1e12), 4.0),
        ("spike1e30", _spike(rng, n, 1e30), 4.0),
        ("tiny", rng.normal(0, 1, size=n) * 1e-30, 3.0e-30),
        ("offset", 1e4 + rng.normal(0, 1, size=n), 4.0),
    ]
    for name, w in [("fp32_1e37", 10), ("fp32_1e37_wide", min(40, n // 2))]:    # 40 x 1e37: prefix sums beyond FLT_MAX
        z = _spike(rng, n, 0.0)
        a = int(rng.integers(0, n - w))
        z[a:a + w] = 1e37 * rng.choice([-1.0, 1.0])
        out.append((name, z, 4.0))
    out.append(("fp32_2e38", _spike(rng, n, 2e38), 4.0))
    out.append(("fp64_1e300", _spike(rng, n, 1e300), 4.0))
    return out


def threshold_at_call(z, min_search=3):
    """Thresholds equal to the first call's exact |value| and the next double below it (both call it: abs < thr is
    False) and the next double above (does not)."""
    _, segs = wc_oracle.segment_region(z, 0.0, min_search)
    v = abs(segs[0][0])
    return [v, np.nextafter(v, 0.0), np.nextafter(v, np.inf)]


CASES = [(name, z, thr) for n, seed in [(40, 1), (77, 2), (130, 3), (180, 4)]
         for name, z, thr in adversarial_regions(n, seed)]


@pytest.mark.parametrize("i", range(len(CASES)), ids=["%s-%d" % (c[0], len(c[1])) for c in CASES])
def test_exact_oracle_matches_full_triangle(i):
    name, z, thr = CASES[i]
    with np.errstate(over="ignore"):
        want = wc_oracle.segment_region(z, thr, 3)
    got = wc_oracle.segment_region_exact(z, thr, 3)
    assert got[0] == want[0]
    assert got[1] == want[1], name


@pytest.mark.parametrize("k", [8, 20])
def test_exact_oracle_chained_spikes(k):
    z = chained_spikes(k)
    want = wc_oracle.segment_region(z, 5.0, 3)
    got = wc_oracle.segment_region_exact(z, 5.0, 3)
    assert len(want[1]) == k and got == want


def test_exact_oracle_threshold_at_a_run_value():
    rng = np.random.default_rng(9)
    for z in [rng.integers(-3, 4, size=60).astype(float), rng.normal(0, 1, size=90), _square_ties(rng, 50)]:
        t_eq, t_below, t_above = threshold_at_call(z)
        for t in (t_eq, t_below, t_above):
            assert wc_oracle.segment_region_exact(z, t, 3) == wc_oracle.segment_region(z, t, 3)
        assert len(wc_oracle.segment_region(z, t_eq, 3)[1]) >= 1


def test_exact_oracle_min_search_and_refusals():
    rng = np.random.default_rng(4)
    z = rng.integers(-2, 3, size=70).astype(float)
    for ms in (0, 1, 5):
        assert wc_oracle.segment_region_exact(z, 2.0, ms) == wc_oracle.segment_region(z, 2.0, ms)
    with pytest.raises(ValueError):
        wc_oracle.segment_region_exact(np.array([1.0, np.nan]), 1.0)
    with pytest.raises(ValueError):                  # every run within the window of a flat region: refuses, not guesses
        wc_oracle.segment_region_exact(np.zeros(2000), -1.0, max_window=1000)
