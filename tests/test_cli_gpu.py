"""GPU: the drop-in command line (wisecondor.py newrefprep/newrefpart/newrefpost/newref/test/testbatch) and the newref
preparation kernels (K1-K3) against what the reference's own CLI produced on the same sample files
(tests/golden/tiny_cli.npz, functions.npz)."""
import os
import sys

import numpy as np
import pytest

import wc_oracle
from wisecondor_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, os.path.join(GOLD))


def _close(a, b, rel=1e-9):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    assert a.shape == b.shape, (a.shape, b.shape)
    ok = (np.isnan(a) & np.isnan(b)) | (a == b) | (np.abs(a - b) <= rel * np.maximum(np.abs(a), np.abs(b)))
    assert ok.all(), "max rel err %g" % np.nanmax(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


def _components_close(a, b):
    for x, y in zip(a, b):
        s = np.sign(np.dot(x, y))
        assert np.max(np.abs(x * s - y)) <= 1e-9 * np.max(np.abs(y))


def _run(argv):
    import wisecondor
    try:
        wisecondor.main(argv)
    except SystemExit as e:
        assert e.code in (0, None), "wisecondor.py %s exited with %s" % (argv[0], e.code)


@pytest.fixture(scope="module")
def tiny():
    return np.load(os.path.join(GOLD, "tiny_cli.npz"), allow_pickle=True)


@pytest.fixture(scope="module")
def fn():
    return np.load(os.path.join(GOLD, "functions.npz"), allow_pickle=True)


@pytest.fixture(scope="module")
def workdir(tmp_path_factory, tiny):
    from make_golden import TINY_BINSIZE, write_sample_npz
    d = tmp_path_factory.mktemp("wc_cli")
    bins = [int(b) for b in tiny['bins']]
    for i in range(tiny['ref_counts'].shape[0]):
        write_sample_npz(str(d / ("r%02d.npz" % i)), tiny['ref_counts'][i], bins, TINY_BINSIZE)
    for t in range(tiny['test_counts'].shape[0]):
        write_sample_npz(str(d / ("t%d.npz" % t)), tiny['test_counts'][t], bins, TINY_BINSIZE)
    # the reference npz exactly as the reference wrote it (arrays from the golden file)
    np.savez_compressed(str(d / "goldref.npz"), arguments={}, runtime={}, binsize=tiny['ref_binsize'],
                        indexes=tiny['ref_indexes'], distances=tiny['ref_distances'],
                        chromosome_sizes=tiny['ref_chromosome_sizes'], mask=tiny['ref_mask'],
                        masked_sizes=tiny['ref_masked_sizes'], pca_components=tiny['ref_pca_components'],
                        pca_mean=tiny['ref_pca_mean'])
    return d


def test_prep_kernels_vs_reference(fn):
    from wisecondor_b200 import wisetools
    bins = list(fn['ingest_bins'])
    samples = [synth.counts_to_sample_dict(fn['ingest_counts'][i], bins, 50000000) for i in range(fn['ingest_counts'].shape[0])]
    masked, chrom_bins, mask = wisetools.toNumpyArray(samples)
    assert np.array_equal(mask, fn['ingest_mask']) and chrom_bins == [len(samples[0][str(c)]) for c in range(1, 23)]
    assert np.array_equal(masked, fn['ingest_masked'])                  # integer / integer-valued total: exact
    corrected, pca = wisetools.trainPCA(masked)
    assert np.array_equal(pca.mean_, fn['ingest_mean'])                 # numpy's summation order on the device
    _close(corrected, fn['ingest_corrected'])
    _components_close(pca.components_, fn['ingest_components'])
    with pytest.raises(ValueError):
        bad = dict(samples[0])
        bad['3'] = bad['3'][:-1]
        wisetools.toNumpyArray([samples[1], bad])


def test_newref_cluster_steps_match_reference(workdir, tiny):
    refs = [str(workdir / ("r%02d.npz" % i)) for i in range(tiny['ref_counts'].shape[0])]
    prep = str(workdir / "ref_prep.npz")
    _run(["newrefprep"] + refs + [prep])
    for part in (1, 2, 3):
        _run(["newrefpart", prep, str(workdir / "ref_part"), str(part), "3", "-refsize", "40"])
    _run(["newrefpost", prep, str(workdir / "ref_part"), "3", str(workdir / "ref.npz")])
    p = np.load(prep, allow_pickle=True)
    assert np.array_equal(p['mask'], tiny['prep_mask'])
    assert np.array_equal(p['maskedChromBins'], tiny['prep_maskedChromBins'])
    assert np.array_equal(p['maskedChromBinSums'], tiny['prep_maskedChromBinSums'])
    assert np.array_equal(p['maskedData'], tiny['prep_maskedData'])
    _close(p['correctedData'], tiny['prep_correctedData'])
    assert p['correctedData'].flags.f_contiguous          # the layout the reference's prep file has
    assert set(p.files) == {'arguments', 'runtime', 'binsize', 'chromosomeBins', 'maskedData', 'mask', 'maskedChromBins',
                            'maskedChromBinSums', 'correctedData', 'pca_components', 'pca_mean'}
    r = np.load(str(workdir / "ref.npz"), allow_pickle=True)
    assert set(r.files) == {'arguments', 'runtime', 'binsize', 'indexes', 'distances', 'chromosome_sizes', 'mask',
                            'masked_sizes', 'pca_components', 'pca_mean'}
    assert r['indexes'].dtype == np.int32 and r['distances'].dtype == np.float64
    assert np.array_equal(r['indexes'], tiny['ref_indexes'])
    _close(r['distances'], tiny['ref_distances'])
    assert np.array_equal(r['chromosome_sizes'], tiny['ref_chromosome_sizes'])
    assert np.array_equal(r['masked_sizes'], tiny['ref_masked_sizes'])
    assert np.array_equal(r['pca_mean'], tiny['ref_pca_mean'])
    _components_close(r['pca_components'], tiny['ref_pca_components'])
    assert r['binsize'].item() == tiny['ref_binsize'].item()
    assert r['arguments'].item()['func'].__name__ == 'toolNewrefPost'
    # distances are bit-identical to the oracle's on the *same* corrected matrix (exact re-score, K6)
    import c_oracle
    mb = [int(b) for b in p['maskedChromBins']]
    oidx, odst = c_oracle.get_reference_rows(p['correctedData'], mb, 0, sum(mb), 40)
    assert np.array_equal(r['indexes'], oidx) and np.array_equal(r['distances'], odst)


def test_newrefprep_with_binsize_matches_reference(workdir, tiny):
    """`newrefprep -binsize 2000000` on 1 Mb samples (scaleSample on every sample before the mask and the PCA,
    wisecondor.py:99-101) against the reference CLI's prep file (tests/golden/tiny_cli_prep_binsize.npz)."""
    gold = np.load(os.path.join(GOLD, "tiny_cli_prep_binsize.npz"), allow_pickle=True)
    refs = [str(workdir / ("r%02d.npz" % i)) for i in range(tiny['ref_counts'].shape[0])]
    prep = str(workdir / "prep2.npz")
    _run(["newrefprep"] + refs + [prep, "-binsize", "2000000"])
    p = np.load(prep, allow_pickle=True)
    assert p['binsize'].item() == gold['binsize'].item() == 2000000
    assert np.array_equal(p['mask'], gold['mask'])
    assert np.array_equal(p['chromosomeBins'], gold['chromosomeBins'])
    assert np.array_equal(p['maskedChromBins'], gold['maskedChromBins'])
    assert np.array_equal(p['maskedChromBinSums'], gold['maskedChromBinSums'])
    assert np.array_equal(p['maskedData'], gold['maskedData'])
    _close(p['correctedData'], gold['correctedData'])


def test_newref_single_command_resumes_and_cleans_up(workdir, tiny):
    refs = [str(workdir / ("r%02d.npz" % i)) for i in range(tiny['ref_counts'].shape[0])]
    out = str(workdir / "whole.npz")
    _run(["newref"] + refs + [out, "-refsize", "40", "-parts", "2"])
    assert not os.path.exists(str(workdir / "whole_prep.npz")) and not os.path.exists(str(workdir / "whole_part_1.npz"))
    r = np.load(out, allow_pickle=True)
    assert np.array_equal(r['indexes'], tiny['ref_indexes'])
    _close(r['distances'], tiny['ref_distances'])


def _check_result(res, tiny, t):
    _close(np.concatenate(list(res['results_z'])), tiny['res%d_z' % t])
    _close(np.concatenate(list(res['results_r'])), tiny['res%d_r' % t])
    _close(res['results_cwz'], tiny['res%d_cwz' % t])
    calls = np.asarray(res['results_calls'], dtype=float).reshape(-1, 5)
    want = tiny['res%d_calls' % t]
    assert calls.shape == want.shape
    assert np.array_equal(calls[:, :3], want[:, :3])                     # chromosome, start bin, end bin: exact
    _close(calls[:, 3:], want[:, 3:])
    _close([res['threshold_z'], res['asdef'], res['aasdef']], tiny['res%d_scalars' % t])
    assert [len(a) for a in res['results_z']] == [int(v) for v in tiny['ref_chromosome_sizes']]


def test_test_tool_matches_reference(workdir, tiny):
    """`test` against the reference npz the reference itself wrote."""
    for t in range(tiny['test_counts'].shape[0]):
        out = str(workdir / ("o%d.npz" % t))
        extra = ["-minrefbins", "10"] + (["-repeats", "3"] if t == 2 else [])
        _run(["test", str(workdir / ("t%d.npz" % t)), out, str(workdir / "goldref.npz")] + extra)
        res = np.load(out, allow_pickle=True)
        assert set(res.files) == {'arguments', 'runtime', 'binsize', 'results_r', 'results_z', 'results_cwz',
                                  'results_calls', 'threshold_z', 'asdef', 'aasdef'}
        _check_result(res, tiny, t)


def test_test_tool_with_mineffectsize_matches_reference(workdir, tiny):
    """`test -mineffectsize 0.25` (wisecondor.py:460 -> fillTriMin) against what the reference's CLI wrote for the same
    files (tests/golden/tiny_cli_mineff.npz, make_golden.golden_cli_tiny_mineff): the filter removes most calls."""
    gold = np.load(os.path.join(GOLD, "tiny_cli_mineff.npz"), allow_pickle=True)
    fewer = 0
    for t in range(tiny['test_counts'].shape[0]):
        out = str(workdir / ("m%d.npz" % t))
        _run(["test", str(workdir / ("t%d.npz" % t)), out, str(workdir / "goldref.npz"), "-minrefbins", "10",
              "-mineffectsize", str(float(gold['mineffectsize']))])
        res = np.load(out, allow_pickle=True)
        _close(np.concatenate(list(res['results_z'])), gold['res%d_z' % t])
        _close(res['results_cwz'], gold['res%d_cwz' % t])
        calls = np.asarray(res['results_calls'], dtype=float).reshape(-1, 5)
        want = gold['res%d_calls' % t]
        assert calls.shape == want.shape, t
        assert np.array_equal(calls[:, :3], want[:, :3])
        _close(calls[:, 3:], want[:, 3:])
        fewer += int(want.shape[0] < tiny['res%d_calls' % t].shape[0])
    assert fewer >= 2


def test_test_tool_flags_and_rescaled_sample_match_reference(workdir, tiny):
    """`test` with -chromosomes / -minzscore / -multitest / -repeats and with a sample binned at half the reference's bin
    size (scaleSample, wisetools.py:20-44) against the reference CLI's own output on the same files
    (tests/golden/tiny_cli_flags.npz, make_golden.golden_cli_tiny_flags)."""
    from make_golden import FLAG_VARIANTS, TINY_BINSIZE, split_counts, write_sample_npz
    gold = np.load(os.path.join(GOLD, "tiny_cli_flags.npz"), allow_pickle=True)
    bins = [int(b) for b in tiny['bins']]
    for name, t, sample_binsize, extra in FLAG_VARIANTS:
        infile = str(workdir / (name + ".npz"))
        if sample_binsize is None:
            write_sample_npz(infile, tiny['test_counts'][t], bins, TINY_BINSIZE)
        else:
            fine, nb = split_counts(tiny['test_counts'][t], bins)
            write_sample_npz(infile, fine, nb, sample_binsize)
        out = str(workdir / (name + "_o.npz"))
        _run(["test", infile, out, str(workdir / "goldref.npz"), "-minrefbins", "10"] + extra)
        res = np.load(out, allow_pickle=True)
        _close(np.concatenate(list(res['results_z'])), gold[name + '_z'])
        _close(np.asarray(res['results_cwz'], dtype=float), gold[name + '_cwz'])
        calls = np.asarray(res['results_calls'], dtype=float).reshape(-1, 5)
        want = gold[name + '_calls']
        assert calls.shape == want.shape, name
        assert np.array_equal(calls[:, :3], want[:, :3]), name
        _close(calls[:, 3:], want[:, 3:])
        _close([res['threshold_z'], res['asdef'], res['aasdef']], gold[name + '_scalars'])


def test_testbatch_equals_single_runs(workdir, tiny):
    outdir = str(workdir / "batch")
    tests = [str(workdir / ("t%d.npz" % t)) for t in (0, 1, 3)]
    _run(["testbatch"] + tests + [outdir, str(workdir / "goldref.npz"), "-minrefbins", "10", "-batch", "2"])
    for t in (0, 1, 3):
        res = np.load(os.path.join(outdir, "t%d.npz" % t), allow_pickle=True)
        _check_result(res, tiny, t)
        single = np.load(str(workdir / ("o%d.npz" % t)), allow_pickle=True)
        assert np.array_equal(np.concatenate(list(res['results_z'])), np.concatenate(list(single['results_z'])), equal_nan=True)
        assert np.array_equal(np.asarray(res['results_calls']), np.asarray(single['results_calls']))


def test_own_reference_then_test_end_to_end(workdir, tiny):
    """newref and test both from this build: calls land where the reference's do."""
    out = str(workdir / "e2e.npz")
    _run(["test", str(workdir / "t1.npz"), out, str(workdir / "ref.npz"), "-minrefbins", "10"])
    res = np.load(out, allow_pickle=True)
    _check_result(res, tiny, 1)


def test_host_only_tools_say_so(workdir):
    import wisecondor
    with pytest.raises(SystemExit) as e:
        wisecondor.main(["convert", "x.bam", "x.npz"])
    assert e.value.code == 2
    assert wc_oracle is not None


def test_config2_shape_prep_and_test_path_vs_oracle():
    """BASELINE configs[1]/[3] shapes at 250 kb (N raw 11 537): normalise + PCA of 600 synthetic samples against the
    oracle's full SVD, then the whole test tool for three samples against the oracle (prefix-sum segmentation oracle:
    the exact triangle is out of reach of a Python double loop at chromosome sizes of ~1000 bins)."""
    from wisecondor_b200 import wisetools
    binsize = 250000
    bins, lam, fac = synth.bin_model(binsize, bin_seed=1)
    ref_counts = synth.sample_counts(600, lam, fac, seed=2)
    test_counts = synth.sample_counts(3, lam, fac, seed=3)
    synth.inject_aberration(test_counts[1], bins, 21, 0.0, 1.0, 1.04, seed=4)
    synth.inject_aberration(test_counts[2], bins, 8, 0.4, 0.5, 0.8, seed=5)
    samples = [synth.counts_to_sample_dict(ref_counts[i], bins, binsize) for i in range(600)]
    masked, chrom_bins, mask = wisetools.toNumpyArray(samples, as_device=True)
    omasked, ochrom_bins, omask = wc_oracle.to_numpy_array(samples)
    assert np.array_equal(mask, omask) and chrom_bins == ochrom_bins
    assert np.array_equal(masked.cpu().numpy(), omasked)
    corrected, pca = wisetools.trainPCA(masked, as_device=True)
    ocorrected, ocomps, omean = wc_oracle.train_pca(omasked)
    assert np.array_equal(pca.mean_, omean)
    _close(corrected.cpu().numpy(), ocorrected)
    _components_close(pca.components_, ocomps)
    # reference-bin search on the device-resident corrected matrix, sampled rows against the C oracle
    import c_oracle
    starts = np.concatenate(([0], np.cumsum(chrom_bins)))
    masked_sizes = [int(mask[starts[i]:starts[i + 1]].sum()) for i in range(22)]
    sums = [int(v) for v in np.cumsum(masked_sizes)]
    idx, dist = wisetools.getReference(corrected, masked_sizes, sums, 100, 1, 1)
    Xh = corrected.cpu().numpy()
    n = Xh.shape[0]
    for r0 in (0, 4000, n - 32):
        oidx, odist = c_oracle.get_reference_rows(Xh, masked_sizes, r0, r0 + 32, 100)
        assert np.array_equal(idx[r0:r0 + 32], oidx) and np.array_equal(dist[r0:r0 + 32], odist)
    ref = dict(binsize=binsize, indexes=idx, distances=dist, chromosome_sizes=np.array(chrom_bins), mask=mask,
               masked_sizes=np.array(masked_sizes), pca_mean=pca.mean_, pca_components=pca.components_)
    tests = [synth.counts_to_sample_dict(test_counts[i], bins, binsize) for i in range(3)]
    thr = 5.0961
    got = wisetools.testSamples(tests, ref, thr, batch=2)
    for t in range(3):
        want = wc_oracle.test_sample(tests[t], binsize, ref, minzscore=thr, segmenter=wc_oracle.segment_region_prefix)
        _close(np.concatenate(got[t]['results_z']), np.concatenate(want['results_z']))
        _close(np.concatenate(got[t]['results_r']), np.concatenate(want['results_r']))
        _close(got[t]['results_cwz'], want['results_cwz'])
        gc = np.asarray(got[t]['results_calls'], dtype=float).reshape(-1, 5)
        wc = np.asarray(want['results_calls'], dtype=float).reshape(-1, 5)
        assert gc.shape == wc.shape and np.array_equal(gc[:, :3], wc[:, :3]), (t, gc, wc)
        _close(gc[:, 3:], wc[:, 3:])
        _close([got[t]['asdef']], [want['asdef']])
    assert len(got[1]['results_calls']) >= 1


def test_newref_on_two_gpus_equals_reference(workdir, tiny):
    """`newref -gpus 2`: one process per GPU, getPart row shards, rows gathered over NCCL (no part files); and the
    `-partfiles` form (host threads + part files, resumable per part).  Same reference file either way."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    refs = [str(workdir / ("r%02d.npz" % i)) for i in range(tiny['ref_counts'].shape[0])]
    out = str(workdir / "two.npz")
    _run(["newref"] + refs + [out, "-refsize", "40", "-gpus", "2"])
    r = np.load(out, allow_pickle=True)
    assert np.array_equal(r['indexes'], tiny['ref_indexes'])
    _close(r['distances'], tiny['ref_distances'])
    assert not os.path.exists(str(workdir / "two_part_1.npz")) and not os.path.exists(str(workdir / "two_prep.npz"))
    out = str(workdir / "twofiles.npz")
    _run(["newref"] + refs + [out, "-refsize", "40", "-gpus", "2", "-parts", "5", "-partfiles"])
    r2 = np.load(out, allow_pickle=True)
    assert np.array_equal(r2['indexes'], r['indexes']) and np.array_equal(r2['distances'], r['distances'])
    assert not os.path.exists(str(workdir / "twofiles_part_3.npz"))


def test_testbatch_on_two_gpus_equals_one(workdir, tiny):
    """`testbatch -gpus 2`: the samples are sharded over two processes / devices; every result file equals the single-GPU one."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    outdir = str(workdir / "batch2")
    tests = [str(workdir / ("t%d.npz" % t)) for t in (0, 1, 3)]
    _run(["testbatch"] + tests + [outdir, str(workdir / "goldref.npz"), "-minrefbins", "10", "-batch", "2", "-gpus", "2"])
    if not os.path.isdir(str(workdir / "batch")):       # (the single-GPU run of test_testbatch_equals_single_runs, when deselected)
        _run(["testbatch"] + tests + [str(workdir / "batch"), str(workdir / "goldref.npz"), "-minrefbins", "10", "-batch", "2"])
    for t in (0, 1, 3):
        res = np.load(os.path.join(outdir, "t%d.npz" % t), allow_pickle=True)
        one = np.load(os.path.join(str(workdir / "batch"), "t%d.npz" % t), allow_pickle=True)
        assert np.array_equal(np.concatenate(list(res['results_z'])), np.concatenate(list(one['results_z'])), equal_nan=True)
        assert np.array_equal(np.asarray(res['results_calls']), np.asarray(one['results_calls']))
        assert float(res['asdef']) == float(one['asdef'])


def test_parts_interchangeable_with_the_reference_workers(workdir, tiny):
    """Cluster mode with mixed workers: the reference's own `newrefpart` (CPU, oracle/_ref) run on THIS build's prep file
    gives bit for bit the part this build computes on the GPU, and a reference of mixed parts assembles with either
    `newrefpost`.  (TEST INFRASTRUCTURE use of oracle/_ref; skipped where it did not travel.)"""
    import subprocess
    ref_cli = os.path.join(ROOT, "oracle", "_ref", "wisecondor.py")
    if not os.path.isfile(ref_cli):
        pytest.skip("oracle/_ref not generated")
    prep = str(workdir / "ref_prep.npz")                     # written by this build in test_newref_cluster_steps...
    assert os.path.isfile(prep)
    r = subprocess.run([sys.executable, ref_cli, "newrefpart", prep, str(workdir / "mix_part"), "2", "3", "-refsize", "40"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-1500:]
    theirs = np.load(str(workdir / "mix_part_2.npz"), allow_pickle=True)
    mine = np.load(str(workdir / "ref_part_2.npz"), allow_pickle=True)
    assert np.array_equal(theirs['indexes'], mine['indexes'])
    assert np.array_equal(theirs['distances'], mine['distances'])          # same prep file -> bit-identical distances
    # assemble: parts 1 and 3 from this build, part 2 from the reference, post-processed by the reference
    import shutil
    shutil.copy(str(workdir / "ref_part_1.npz"), str(workdir / "mix_part_1.npz"))
    shutil.copy(str(workdir / "ref_part_3.npz"), str(workdir / "mix_part_3.npz"))
    r = subprocess.run([sys.executable, ref_cli, "newrefpost", prep, str(workdir / "mix_part"), "3", str(workdir / "mix.npz")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-1500:]
    mixed = np.load(str(workdir / "mix.npz"), allow_pickle=True)
    whole = np.load(str(workdir / "ref.npz"), allow_pickle=True)
    for key in ("indexes", "distances", "mask", "masked_sizes", "chromosome_sizes", "pca_mean", "pca_components"):
        assert np.array_equal(mixed[key], whole[key]), key


def test_parts_on_the_reference_prep_file_match_reference(workdir, tiny):
    """This build's `newrefpart` and `newrefpost` on the prep file the reference's own `newrefprep` wrote (rebuilt from its
    arrays in tests/golden/tiny_cli.npz): part 2 of 3 holds bit for bit the reference's rows of that part, and the
    assembled reference file equals the one the reference's `newrefpost` wrote from its three parts."""
    prep = str(workdir / "goldprep.npz")
    np.savez_compressed(prep, arguments={}, runtime={}, binsize=tiny['binsize'], chromosomeBins=tiny['ref_chromosome_sizes'],
                        maskedData=tiny['prep_maskedData'], mask=tiny['prep_mask'],
                        maskedChromBins=tiny['prep_maskedChromBins'], maskedChromBinSums=tiny['prep_maskedChromBinSums'],
                        correctedData=np.asfortranarray(tiny['prep_correctedData']),
                        pca_components=tiny['ref_pca_components'], pca_mean=tiny['ref_pca_mean'])
    for part in (1, 2, 3):
        _run(["newrefpart", prep, str(workdir / "gold_part"), str(part), "3", "-refsize", "40"])
    a, b = wc_oracle.get_part(1, 3, tiny['ref_indexes'].shape[0])
    mine = np.load(str(workdir / "gold_part_2.npz"), allow_pickle=True)
    assert np.array_equal(mine['indexes'], tiny['ref_indexes'][a:b])
    assert np.array_equal(mine['distances'], tiny['ref_distances'][a:b])
    _run(["newrefpost", prep, str(workdir / "gold_part"), "3", str(workdir / "gold.npz")])
    r = np.load(str(workdir / "gold.npz"), allow_pickle=True)
    for key in ("indexes", "distances", "chromosome_sizes", "mask", "masked_sizes", "pca_mean", "pca_components"):
        assert np.array_equal(r[key], tiny['ref_' + key]), key
    assert r['binsize'].item() == tiny['ref_binsize'].item()


def test_reference_consumers_read_our_results(workdir, tiny):
    """The reference's own `report` tool (a pure consumer of sample + result npz, wisecondor.py:304-342) and its `test`
    tool accept the files this build writes."""
    import subprocess
    ref_cli = os.path.join(ROOT, "oracle", "_ref", "wisecondor.py")
    if not os.path.isfile(ref_cli):
        pytest.skip("oracle/_ref not generated")
    out = str(workdir / "o1.npz")                            # this build's result for test sample 1
    assert os.path.isfile(out)
    r = subprocess.run([sys.executable, ref_cli, "report", str(workdir / "t1.npz"), out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-1500:]
    assert "z-score" in r.stdout.lower() or "chr" in r.stdout.lower() or len(r.stdout) > 50
    # the reference's test tool on the reference file THIS build wrote
    r = subprocess.run([sys.executable, ref_cli, "test", str(workdir / "t1.npz"), str(workdir / "theirs_on_ours.npz"),
                        str(workdir / "ref.npz"), "-minrefbins", "10"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-1500:]
    res = np.load(str(workdir / "theirs_on_ours.npz"), allow_pickle=True)
    _check_result(res, tiny, 1)
