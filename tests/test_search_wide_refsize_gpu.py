"""The wide-refsize reference-bin search (wc_newref_topk_wide, refsize up to 4096) against the C oracle: indexes
identical and distances bit-identical, on every row searched.

Covers refsizes 385 ... 4096 on small and medium genomes (rows with fewer candidates than refsize get fillers), degenerate
chromosome layouts, odd and tiny sample counts, a matrix outside fp16's range, row ranges and getPart parts, a 50 kb
matrix with 600 samples on sampled row ranges, the adversarial families of test_search_adversarial_inputs at refsize
600 (near-tie clusters, the 1e10 cut, NaN and +-inf), a plateau of bit-equal distances wider than refsize, equality
with the narrow entry where both run, the refusal above 4096, and the command line (`newref -refsize 600` single,
with -parts and on two GPUs, then `test` / `testbatch` on that reference)."""
import os
import sys

import numpy as np
import pytest

import c_oracle
import wc_oracle
from test_search_adversarial_inputs import MID_BINS, near_tie, range_boundary, low_rank, pivot_starved
from wisecondor_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLD)

MEDIUM_BINS = [int(b) for b in np.maximum(1, np.array(synth.chrom_bins(250000)) // 4)]


def _wide(X, bins, r0, r1, k):
    import torch
    from wisecondor_b200 import device
    x = torch.from_numpy(np.ascontiguousarray(X, dtype=np.float64)).cuda()
    idx, dist = device.newref_topk_wide(x, bins, r0, r1, k)
    return idx.cpu().numpy(), dist.cpu().numpy()


def _assert_same(idx, dist, oidx, odist):
    assert idx.shape == oidx.shape and dist.shape == odist.shape
    bad = np.flatnonzero((idx != oidx).any(axis=1))
    assert bad.size == 0, "index rows differ: %s (first: %s vs %s)" % (bad[:8], idx[bad[0]][:10], oidx[bad[0]][:10])
    assert np.array_equal(dist.view(np.int64), odist.view(np.int64)), "distances not bit-identical"


def _check(X, bins, r0, r1, k):
    oidx, odist = c_oracle.get_reference_rows(X, bins, r0, r1, k)
    idx, dist = _wide(X, bins, r0, r1, k)
    _assert_same(idx, dist, oidx, odist)
    return oidx


@pytest.mark.parametrize("k", [385, 447, 512, 513, 1000, 2048, 4096])
def test_small_and_medium_genomes(small_bins, k):
    X = synth.corrected_like(small_bins, 40, seed=k)
    oidx = _check(X, small_bins, 0, X.shape[0], k)
    assert (oidx == -1).any() == (k > X.shape[0] - max(small_bins))
    X = synth.corrected_like(MEDIUM_BINS, 64, seed=k + 1)
    oidx = _check(X, MEDIUM_BINS, 0, X.shape[0], k)
    assert (oidx[:, -1] == -1).any() == (k > X.shape[0] - max(MEDIUM_BINS))


def test_degenerate_genomes():
    X = synth.corrected_like([25], 10, seed=1)
    idx, dist = _wide(X, [25], 0, 25, 500)
    assert (idx == -1).all() and (dist == 1e10).all()
    bins = [0, 9, 0, 0, 14, 3, 0]
    X = synth.corrected_like(bins, 7, seed=2)
    _check(X, bins, 0, 26, 400)
    _check(X, bins, 3, 20, 1)
    bins = [40, 35, 30, 500]
    _check(synth.corrected_like(bins, 33, seed=4), bins, 0, 605, 385)


@pytest.mark.parametrize("S", [1, 3, 7, 37, 129])
def test_odd_and_small_sample_counts(S):
    X = synth.corrected_like(MEDIUM_BINS, S, seed=S)
    _check(X, MEDIUM_BINS, 0, X.shape[0], 700)


def test_matrix_outside_fp16_range():
    X = synth.corrected_like(MEDIUM_BINS, 48, seed=9)
    X[100:140] += 1e5 * np.random.default_rng(0).standard_normal((40, 48))
    X[500, 3] = 1.0 + 70000.0
    _check(X, MEDIUM_BINS, 0, X.shape[0], 600)


def test_row_ranges_and_parts_concatenate_to_whole():
    from wisecondor_b200 import wisetools
    X = synth.corrected_like(MEDIUM_BINS, 30, seed=5)
    n = X.shape[0]
    for r0, r1 in ((0, 1), (1, 130), (127, 129), (n - 200, n), (700, 700)):
        _check(X, MEDIUM_BINS, r0, r1, 600)
    sums = list(np.cumsum(MEDIUM_BINS))
    whole_i, whole_d = wisetools.getReference(X, MEDIUM_BINS, sums, 600, 1, 1)       # host array: uploaded through _mem
    oidx, odist = c_oracle.get_reference_rows(X, MEDIUM_BINS, 0, n, 600)
    _assert_same(whole_i, whole_d, oidx, odist)
    for parts in (3, 7):
        got = [wisetools.getReference(X, MEDIUM_BINS, sums, 600, p, parts) for p in range(1, parts + 1)]
        assert np.array_equal(np.concatenate([g[0] for g in got]), whole_i)
        assert np.array_equal(np.concatenate([g[1] for g in got]), whole_d)


def test_50kb_600_samples_sampled_rows():
    bins = synth.chrom_bins(50000)
    X = synth.corrected_like(bins, 600, seed=21)
    n = X.shape[0]
    rng = np.random.default_rng(3)
    for r0 in [0, n - 48] + sorted(rng.choice(n - 48, 3, replace=False).tolist()):
        _check(X, bins, int(r0), int(r0) + 48, 1000)


@pytest.mark.parametrize("M,delta", [(599, 1e-7), (600, 1e-9), (601, 1e-5), (900, 1e-7)])
def test_near_tie_clusters(M, delta):
    c = near_tie(M, delta, k=600, bins=[3 * b for b in MID_BINS[:4]] + MID_BINS[4:])
    _check(c["X"], c["bins"], 0, c["X"].shape[0], 600)


@pytest.mark.parametrize("S", [1, 8])
def test_1e10_cut_nan_and_inf(S):
    c = range_boundary(S)
    _check(c["X"], c["bins"], 0, c["X"].shape[0], 600)


def test_low_rank_and_duplicate_rows():
    c = low_rank(3, k=600)
    _check(c["X"], c["bins"], 0, c["X"].shape[0], 600)
    c = pivot_starved(k=600, zero_rows=40)
    _check(c["X"], c["bins"], 0, c["X"].shape[0], 600)


def test_tie_plateau_wider_than_refsize():
    """Target bins on chromosome 4 with 1500 candidates at one bit-equal distance a^2 (x_t +- a e_s, a = 2^-6, x_t on a
    2^-10 grid) spread over chromosomes 1-3: the first 600 by bin index must win, in index order."""
    S, a = 800, 2.0 ** -6
    bins = [600, 500, 700, 60]
    rng = np.random.default_rng(11)
    X = 1.0 + rng.normal(0.0, 0.3, size=(sum(bins), S))
    t0 = sum(bins[:3])
    for t in (t0, t0 + 7, t0 + 59):
        X[t] = 1.0 + np.round(rng.normal(0.0, 0.05, S) * 1024) / 1024
    shell = np.sort(rng.choice(t0, 1500, replace=False))
    which = rng.choice(2 * S, 1500, replace=False)
    for r, w in zip(shell, which):
        X[r] = X[t0]
        X[r, w % S] += a if w < S else -a
    oidx = _check(X, bins, t0, t0 + 1, 600)
    assert np.array_equal(oidx[0], shell[:600])
    _check(X, bins, t0, sum(bins), 2000)


@pytest.mark.parametrize("k", [1, 100, 384])
def test_wide_equals_narrow(k):
    import torch
    from wisecondor_b200 import device
    X = synth.corrected_like(MEDIUM_BINS, 50, seed=k)
    x = torch.from_numpy(X).cuda()
    n = X.shape[0]
    ni, nd = device.newref_topk(x, MEDIUM_BINS, 0, n, k)
    wi, wd = device.newref_topk_wide(x, MEDIUM_BINS, 0, n, k)
    _assert_same(wi.cpu().numpy(), wd.cpu().numpy(), ni.cpu().numpy(), nd.cpu().numpy())
    si, sd = device.newref_search(x, MEDIUM_BINS, 0, n, k)
    _assert_same(si.cpu().numpy(), sd.cpu().numpy(), ni.cpu().numpy(), nd.cpu().numpy())


def test_refsize_bounds_refused():
    import torch
    from wisecondor_b200 import _cabi, device
    X = synth.corrected_like([40, 35], 8, seed=1)
    x = torch.from_numpy(X).cuda()
    for k in (0, 4097):
        with pytest.raises(_cabi.WisecondorError):
            device.newref_topk_wide(x, [40, 35], 0, 75, k)
        with pytest.raises(_cabi.WisecondorError):
            device.newref_search(x, [40, 35], 0, 75, k)
    with pytest.raises(_cabi.WisecondorError):
        device.newref_topk_wide(x, [40, 30], 0, 75, 500)       # chromosome sizes do not add up to N
    _check(X, [40, 35], 0, 75, 4096)


def _run(argv):
    import wisecondor
    try:
        wisecondor.main(argv)
    except SystemExit as e:
        assert e.code in (0, None), "wisecondor.py %s exited with %s" % (argv[0], e.code)


def _close(a, b, rel=1e-9):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    assert a.shape == b.shape, (a.shape, b.shape)
    ok = (np.isnan(a) & np.isnan(b)) | (a == b) | (np.abs(a - b) <= rel * np.maximum(np.abs(a), np.abs(b)))
    assert ok.all(), "max rel err %g" % np.nanmax(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


def _check_vs_oracle(res, want):
    _close(np.concatenate(list(res['results_z'])), np.concatenate(want['results_z']))
    _close(np.concatenate(list(res['results_r'])), np.concatenate(want['results_r']))
    _close(res['results_cwz'], want['results_cwz'])
    gc = np.asarray(res['results_calls'], dtype=float).reshape(-1, 5)
    wc = np.asarray(want['results_calls'], dtype=float).reshape(-1, 5)
    assert gc.shape == wc.shape and np.array_equal(gc[:, :3], wc[:, :3]), (gc, wc)
    _close(gc[:, 3:], wc[:, 3:])


def test_cli_newref_refsize_600_then_test_and_testbatch(tmp_path):
    """`newref -refsize 600` on the four tiny reference samples, single run, with -parts 3 and (two GPUs) -gpus 2: the C
    oracle's rows on the prep's corrected matrix; `test` and `testbatch` on that reference against wc_oracle."""
    import torch
    from make_golden import TINY_BINSIZE, write_sample_npz
    tiny = np.load(os.path.join(GOLD, "tiny_cli.npz"), allow_pickle=True)
    bins = [int(b) for b in tiny['bins']]
    refs = []
    for i in range(tiny['ref_counts'].shape[0]):
        refs.append(str(tmp_path / ("r%02d.npz" % i)))
        write_sample_npz(refs[-1], tiny['ref_counts'][i], bins, TINY_BINSIZE)
    nt = tiny['test_counts'].shape[0]
    for t in range(nt):
        write_sample_npz(str(tmp_path / ("t%d.npz" % t)), tiny['test_counts'][t], bins, TINY_BINSIZE)
    prep = str(tmp_path / "prep.npz")
    _run(["newrefprep"] + refs + [prep])
    p = np.load(prep, allow_pickle=True)
    mb = [int(b) for b in p['maskedChromBins']]
    oidx, odist = c_oracle.get_reference_rows(p['correctedData'], mb, 0, sum(mb), 600)
    assert oidx.shape == (672, 600)
    out_ref = str(tmp_path / "ref.npz")
    runs = [[], ["-parts", "3"]] + ([["-gpus", "2"]] if torch.cuda.device_count() >= 2 else [])
    for extra in runs:
        out = str(tmp_path / ("ref%d.npz" % len(extra)))
        _run(["newref"] + refs + [out, "-refsize", "600"] + extra)
        r = np.load(out, allow_pickle=True)
        assert np.array_equal(r['indexes'], oidx), extra
        assert np.array_equal(r['distances'], odist), extra
        if not extra:
            os.replace(out, out_ref)
    r = np.load(out_ref, allow_pickle=True)
    ref = {key: r[key] for key in ('indexes', 'distances', 'chromosome_sizes', 'mask', 'masked_sizes', 'pca_mean',
                                   'pca_components')}
    ref['binsize'] = r['binsize'].item()
    wants = []
    for t in range(nt):
        sample = synth.counts_to_sample_dict(tiny['test_counts'][t], bins, TINY_BINSIZE)
        wants.append(wc_oracle.test_sample(sample, TINY_BINSIZE, ref, minrefbins=10))
        out = str(tmp_path / ("o%d.npz" % t))
        _run(["test", str(tmp_path / ("t%d.npz" % t)), out, out_ref, "-minrefbins", "10"])
        _check_vs_oracle(np.load(out, allow_pickle=True), wants[t])
    outdir = str(tmp_path / "batch")
    _run(["testbatch"] + [str(tmp_path / ("t%d.npz" % t)) for t in range(nt)] + [outdir, out_ref, "-minrefbins", "10",
                                                                                  "-batch", "3"])
    for t in range(nt):
        _check_vs_oracle(np.load(os.path.join(outdir, "t%d.npz" % t), allow_pickle=True), wants[t])


def test_symmetric_shards_refuse_wide_refsize():
    import torch
    from wisecondor_b200 import shard
    with pytest.raises(ValueError):
        shard.ShardedSearch(1000, 8, 385, 0, 1, torch.device("cuda", 0), symmetric=True)
