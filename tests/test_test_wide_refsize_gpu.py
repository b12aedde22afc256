"""The test path with refsize above 512 (K8w, wc_zscore_wide_kernel / wc_zscore_wide_pairs_kernel) against
wc_oracle, on every sample: z, r, refsizes bit-identical (NaN-equal) and the sigma average equal.

Covers refsizes on both sides of numpy's split edges (513 ... 4096, and one at or above N - N_c so that the (-1, 1e10)
fillers and the cutoff take part), batches of 1 to 64 samples, NaN / +-inf / negative / +-0 test values in the most
used reference bins, pre-marked working copies, both later-pass kernels (dirty-pair list and full pass), kept counts
exactly at 128 * 2^m + {-1, 0, 1, 7, 8}, the N x stride < 2^31 refusal, and the whole `test` / `testbatch` tools on a
reference assembled by `newrefpost` from part files with refsize 600."""
import ctypes
import os
import sys

import numpy as np
import pytest

import c_oracle
import wc_oracle
from test_test_path_edges_gpu import _global_table, _passes
from wisecondor_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLD)


def _upload(tests, copy0, B, n):
    import torch
    from wisecondor_b200 import device
    ldb = device.pad32(B)
    T = torch.ones((n, ldb), dtype=torch.float64, device="cuda")
    C = torch.ones((n, ldb), dtype=torch.float64, device="cuda")
    T[:, :B] = torch.from_numpy(np.ascontiguousarray(tests.T)).cuda()
    C[:, :B] = torch.from_numpy(np.ascontiguousarray(copy0.T)).cuda()
    return T, C


def _assert_sample(b, got, want):
    z, r, sizes, asdef = got
    assert np.array_equal(z[b], want[0], equal_nan=True), "sample %d z" % b
    assert np.array_equal(r[b], want[1], equal_nan=True), "sample %d r" % b
    assert np.array_equal(sizes[b], want[2]), "sample %d refsizes" % b
    assert asdef[b] == want[3] or (np.isnan(asdef[b]) and np.isnan(want[3])), "sample %d sigma" % b


# 250 kb chromosome shape / 4: N = 2 877 bins, the largest chromosome has 249, so refsize 4096 >= N - N_c gets fillers
@pytest.mark.parametrize("B,k,regime", [(31, 513, "few"), (33, 520, "many"), (1, 1000, "many"), (64, 1024, "few"),
                                        (33, 1025, "many"), (31, 1031, "few"), (1, 2048, "many"), (33, 2049, "many"),
                                        (31, 4096, "many")])
def test_k8w_every_sample_special_values_and_both_later_pass_kernels(B, k, regime):
    """As test_k8_every_sample_special_values_and_both_later_pass_kernels, at refsizes above 512: every sample against
    repeat_test from its (partly pre-marked) copy, and the device's per-pass pair counts against the dirty set modelled
    from the oracle's marks and the usage table."""
    from wisecondor_b200 import device
    bins = [int(b) for b in np.maximum(3, np.array(synth.chrom_bins(250000)) // 4)]
    n = sum(bins)
    sums = list(np.cumsum(bins))
    X = synth.corrected_like(bins, 16, seed=B + k)
    idx, dst = c_oracle.get_reference_rows(X, bins, 0, n, k)
    if k >= n - max(bins):
        assert (idx == -1).any() and (dst == 1e10).any()              # fillers on the largest chromosomes
    cutoff = wc_oracle.get_optimal_cutoff(dst, 3)
    use = _global_table(idx, dst, bins, cutoff)
    assert use.sum(axis=1).max() > 512
    hot = np.argsort(-use.sum(axis=0), kind="stable")[:24]
    rng = np.random.default_rng(B * 1000 + k)
    tests = 1.0 + rng.normal(0, 0.03, size=(B, n))
    few = regime == "few"
    thr = 5.0 if few else 1.2
    specials = [np.nan, np.inf, -np.inf, -1.0, -0.5, -0.0, 0.0]
    for b in range(B):
        a = int(rng.integers(0, n - 40))
        tests[b, a:a + int(rng.integers(3, 40))] *= rng.choice([0.97, 1.03] if few else [0.8, 1.2])
        if not few or b in (0, B - 1):
            for j, v in enumerate(specials):
                tests[b, hot[(b + 3 * j) % len(hot)]] = v
    copy0 = np.copy(tests)
    for b in range(0, B, 2):
        copy0[b, rng.random(n) < 0.05] = -1.0
        copy0[b, hot[b % len(hot)]] = -1.0
    repeats = 4
    T, C = _upload(tests, copy0, B, n)
    table = device.ReferenceTable(idx, dst, bins, cutoff)
    got = device.zscore_batch(T, B, table, thr, repeats, copy_init=C)
    pairs = device.last_test_stats()["zscore_pairs_per_pass"]
    got = [g.cpu().numpy() for g in got]

    newly = np.zeros((repeats, n, B), dtype=bool)
    for b in range(B):
        outs, copies = _passes(tests[b], copy0[b], idx, dst, bins, sums, cutoff, thr, repeats)
        _assert_sample(b, got, outs[-1])
        for p in range(1, repeats):
            newly[p, :, b] = (copies[p] == -1.0) & (copies[p - 1] != -1.0)
    limit = n * B // 8
    kinds = []
    for p in range(1, repeats):
        dirty = int((use.astype(np.int32) @ newly[p].astype(np.int32) > 0).sum())
        assert pairs[p] == (dirty if dirty <= limit else n * B), "pass %d: %d dirty pairs, device %d" % (p, dirty, pairs[p])
        kinds.append("pairs" if dirty <= limit else "full")
    if few:
        assert "pairs" in kinds and any(pairs[p] > 0 for p in range(1, repeats))
    else:
        assert "full" in kinds


def _edge_counts():
    return [128 * 2 ** m + d for m in range(6) for d in (-1, 0, 1, 7, 8)]


def test_k8w_kept_counts_on_the_split_edges():
    """One target bin per sample whose kept count is exactly 128 * 2^m + {-1, 0, 1, 7, 8} (m = 0..5): the copy marks
    the right number of its reference bins.  The table is synthetic (distinct other-chromosome bins per row, every
    distance below the cutoff), so count = refsize = 4104 for every bin; one pass and then two more from the marks."""
    from wisecondor_b200 import device
    bins = [int(b) for b in np.maximum(3, np.array(synth.chrom_bins(250000)) // 2)]
    n = sum(bins)
    sums = list(np.cumsum(bins))
    k = 4104
    rng = np.random.default_rng(7)
    idx = np.empty((n, k), dtype=np.int32)
    starts = np.concatenate(([0], np.cumsum(bins)))
    for c in range(len(bins)):
        nother = n - bins[c]
        for i in range(starts[c], starts[c + 1]):
            idx[i] = rng.choice(nother, size=k, replace=False)
    dst = np.sort(rng.random((n, k)), axis=1)
    cutoff = 2.0
    targets = _edge_counts()
    B = len(targets)
    tests = 1.0 + rng.normal(0, 0.03, size=(B, n))
    copy0 = np.copy(tests)
    use = _global_table(idx, dst, bins, cutoff)
    tbin = rng.choice(n, size=B, replace=False)
    for b, t in enumerate(targets):
        refs = np.flatnonzero(use[tbin[b]])
        assert len(refs) == k
        copy0[b, rng.choice(refs, size=k - t, replace=False)] = -1.0
    T, C = _upload(tests, copy0, B, n)
    table = device.ReferenceTable(idx, dst, bins, cutoff)
    for repeats, thr in ((1, 4.0), (3, 1.0)):
        got = [g.cpu().numpy() for g in device.zscore_batch(T, B, table, thr, repeats, copy_init=C)]
        for b, t in enumerate(targets):
            outs, _ = _passes(tests[b], copy0[b], idx, dst, bins, sums, cutoff, thr, repeats)
            if repeats == 1:
                assert got[2][b, tbin[b]] == t
            _assert_sample(b, got, outs[-1])


def test_table_size_limit_is_refused_before_any_memory_is_touched():
    """N x wc_table_stride(k) must stay below 2^31 (int32 table, reverse-table offsets and pair codes): at 50 kb
    (N = 57 633) refsize 37 260 is the largest accepted, 37 261 is refused by wc_zscore_batch, wc_test_table and
    ReferenceTable.  Only argument values reach the library: the pointers are never dereferenced."""
    from wisecondor_b200 import _cabi, device
    L = _cabi.lib()
    n = int(sum(synth.chrom_bins(50000)))
    assert n == 57633
    assert n * L.wc_table_stride(37260) < 2 ** 31 <= n * L.wc_table_stride(37261)
    ctx = _cabi.context(0)
    fake = ctypes.c_void_p(4096)                       # never dereferenced: the check comes first
    rc = L.wc_zscore_batch(ctx.handle, fake, None, n, 32, 32, fake, fake, fake, fake, 37261, 4.0, 5, fake, fake, fake,
                           fake, None)
    assert rc != 0 and "2^31" in L.wc_last_error().decode()
    bins = np.ascontiguousarray(synth.chrom_bins(50000), dtype=np.int32)
    rc = L.wc_test_table(ctx.handle, fake, fake, n, 37261, bins.ctypes.data_as(ctypes.c_void_p), len(bins), 1.0, fake,
                         fake, fake, fake, None)
    assert rc != 0 and "2^31" in L.wc_last_error().decode()
    wide_idx = np.broadcast_to(np.int32(0), (n, 37261))        # shape only: nothing of this size is allocated
    wide_dst = np.broadcast_to(np.float64(0), (n, 37261))
    with pytest.raises(_cabi.WisecondorError, match="2\\^31"):
        device.ReferenceTable(wide_idx, wide_dst, synth.chrom_bins(50000), 1.0)


# ---- the command line on a reference with refsize 600 ----------------------------------------------------------------
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
    _close([res['threshold_z'], res['asdef'], res['aasdef']], [want['threshold_z'], want['asdef'], want['aasdef']])


def test_cli_test_and_testbatch_on_parts_with_refsize_600(tmp_path):
    """Part files in the reference's schema with refsize 600 (the C oracle's rows, as the reference's own `newrefpart`
    writes them; above this build's search limit of 384), joined by this build's `newrefpost`; `test` and `testbatch`
    on the four tiny samples against wc_oracle.test_sample."""
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
    n = sum(mb)
    assert n == 672
    for part in range(3):
        a, b = wc_oracle.get_part(part, 3, n)
        idx, dst = c_oracle.get_reference_rows(p['correctedData'], mb, a, b, 600)
        np.savez_compressed(str(tmp_path / ("part_%d.npz" % (part + 1))), arguments={}, runtime={}, indexes=idx,
                            distances=dst)
    out_ref = str(tmp_path / "ref.npz")
    _run(["newrefpost", prep, str(tmp_path / "part"), "3", out_ref])
    r = np.load(out_ref, allow_pickle=True)
    assert r['indexes'].shape == (672, 600)
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
    assert max(int(np.max(w['_sizes'])) for w in wants) > 512
    outdir = str(tmp_path / "batch")
    _run(["testbatch"] + [str(tmp_path / ("t%d.npz" % t)) for t in range(nt)] + [outdir, out_ref, "-minrefbins", "10",
                                                                                  "-batch", "3"])
    for t in range(nt):
        _check_vs_oracle(np.load(os.path.join(outdir, "t%d.npz" % t), allow_pickle=True), wants[t])


def test_250kb_shape_test_path_with_refsize_1000_vs_oracle():
    """test_config2_shape_prep_and_test_path_vs_oracle's 250 kb shape (N raw 11 537) with a refsize-1000 reference
    from the C oracle on this build's corrected matrix: the whole test tool for three samples against the oracle."""
    from wisecondor_b200 import wisetools
    binsize = 250000
    bins, lam, fac = synth.bin_model(binsize, bin_seed=1)
    ref_counts = synth.sample_counts(200, lam, fac, seed=2)
    test_counts = synth.sample_counts(3, lam, fac, seed=3)
    synth.inject_aberration(test_counts[1], bins, 21, 0.0, 1.0, 1.04, seed=4)
    synth.inject_aberration(test_counts[2], bins, 8, 0.4, 0.5, 0.8, seed=5)
    samples = [synth.counts_to_sample_dict(ref_counts[i], bins, binsize) for i in range(200)]
    masked, chrom_bins, mask = wisetools.toNumpyArray(samples, as_device=True)
    corrected, pca = wisetools.trainPCA(masked, as_device=True)
    starts = np.concatenate(([0], np.cumsum(chrom_bins)))
    masked_sizes = [int(mask[starts[i]:starts[i + 1]].sum()) for i in range(22)]
    Xh = np.ascontiguousarray(corrected.cpu().numpy())
    idx, dist = c_oracle.get_reference_rows(Xh, masked_sizes, 0, Xh.shape[0], 1000)
    ref = dict(binsize=binsize, indexes=idx, distances=dist, chromosome_sizes=np.array(chrom_bins), mask=mask,
               masked_sizes=np.array(masked_sizes), pca_mean=pca.mean_, pca_components=pca.components_)
    tests = [synth.counts_to_sample_dict(test_counts[i], bins, binsize) for i in range(3)]
    thr = 5.0961
    got = wisetools.testSamples(tests, ref, thr, batch=2)
    for t in range(3):
        want = wc_oracle.test_sample(tests[t], binsize, ref, minzscore=thr, segmenter=wc_oracle.segment_region_prefix)
        assert int(np.max(want['_sizes'])) > 512
        _close(np.concatenate(got[t]['results_z']), np.concatenate(want['results_z']))
        _close(np.concatenate(got[t]['results_r']), np.concatenate(want['results_r']))
        _close(got[t]['results_cwz'], want['results_cwz'])
        gc = np.asarray(got[t]['results_calls'], dtype=float).reshape(-1, 5)
        wc = np.asarray(want['results_calls'], dtype=float).reshape(-1, 5)
        assert gc.shape == wc.shape and np.array_equal(gc[:, :3], wc[:, :3]), (t, gc, wc)
        _close(gc[:, 3:], wc[:, 3:])
        _close([got[t]['asdef']], [want['asdef']])
    assert len(got[1]['results_calls']) >= 1
