"""CPU: wc_oracle.pairwise_sum and mean_std_model equal numpy's np.sum / np.mean / np.std bit for bit at the lengths
the wide-refsize z-score kernels (K8w) sum: 513 to 37 000 values, numpy's split edges 128 * 2^m + {-1, 0, 1, 7, 8}
among them, on plain arrays and on compacted copies `a[a >= 0]` as trySample builds them (wisetools.py:425)."""
import numpy as np
import pytest

import wc_oracle

EDGES = [128 * 2 ** m + d for m in range(2, 9) for d in (-1, 0, 1, 7, 8)]
LENGTHS = sorted(set([513, 520, 1000, 1024, 1025, 1031, 2048, 2049, 4096, 8191, 8192, 8193, 37000] + EDGES))


@pytest.mark.parametrize("n", LENGTHS)
def test_pairwise_sum_and_mean_std_equal_numpy(n):
    rng = np.random.default_rng(n)
    a = (1.0 + rng.normal(0, 0.05, size=n)) * 10.0 ** rng.integers(-3, 4, size=n)
    assert wc_oracle.pairwise_sum(a) == np.sum(a)
    m, sd = wc_oracle.mean_std_model(a)
    assert m == np.mean(a) and sd == np.std(a)


@pytest.mark.parametrize("n", [600, 1031, 4104, 8200, 37000])
def test_compacted_copies_equal_numpy(n):
    """Dropping marked (-1), negative and NaN values changes the length and so the split tree: the model of the kept
    array must still be numpy's."""
    rng = np.random.default_rng(n + 1)
    a = 1.0 + rng.normal(0, 0.05, size=n)
    for frac in (0.001, 0.1, 0.5):
        b = np.copy(a)
        drop = rng.random(n) < frac
        b[drop] = rng.choice([-1.0, -0.5, np.nan, -np.inf], size=int(drop.sum()))
        b[rng.choice(np.flatnonzero(~drop))] = -0.0     # kept: -0.0 >= 0
        kept = b[b >= 0]
        assert len(kept) == n - int(drop.sum())
        assert wc_oracle.pairwise_sum(kept) == np.sum(kept)
        m, sd = wc_oracle.mean_std_model(kept)
        assert m == np.mean(kept) and sd == np.std(kept)
