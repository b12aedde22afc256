#!/usr/bin/env python
"""TEST INFRASTRUCTURE - regenerates the golden vectors in tests/golden/ by running the REFERENCE ITSELF.

The reference (VUmcCGP/wisecondor) ships no tests or fixtures, so the pins are outputs of its own code executed
in the build container: oracle/make_ref.py writes a mechanically converted Python-3 copy to oracle/_ref/
(git-ignored), and this script drives it

  * end to end through its CLI (`wisecondor.py newref` / `test`) on seeded synthetic sample npz files, and
  * function by function (wisetools.getRefForBins/getReference, trySample/repeatTest, getOptimalCutoff,
    fillTri/fillTriMin + TriArr.segmentTri, toNumpyArray/toNumpyRefFormat/trainPCA/applyPCA, scaleSample)

and stores inputs + outputs as small compressed npz files.  Only data is committed, never reference code.
Run from the repo root in the build container (needs /root/reference):  python tests/golden/make_golden.py
"""
import contextlib
import io
import json
import os
import shutil
import subprocess
import sys
import tempfile
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.path.join(ROOT, "oracle", "_ref")
sys.path.insert(0, ROOT)

from wisecondor_b200 import synth  # noqa: E402

TINY_BINS = [60, 55, 50, 48, 45, 43, 40, 37, 36, 34, 34, 33, 29, 27, 26, 23, 20, 20, 15, 16, 12, 13]
TINY_BINSIZE = 1000000


def write_sample_npz(path, row, bins, binsize):
    """A sample npz with the keys convert writes (wisecondor.py:22-26); X/Y are present but unused."""
    s = {}
    pos = 0
    for c, n in zip(synth.AUTOSOMES, bins):
        s[c] = np.ascontiguousarray(row[pos:pos + n]).astype(np.int32)
        pos += n
    s['X'] = np.zeros(5, dtype=np.int32)
    s['Y'] = np.zeros(3, dtype=np.int32)
    quality = {key: 0 for key in ('mapped', 'unmapped', 'no_coordinate', 'filter_rmdup', 'filter_mapq', 'pre_retro',
                                  'post_retro', 'pair_fail')}          # the keys convert writes (wisetools.py:209-216)
    np.savez_compressed(path, arguments={'binsize': float(binsize)}, runtime={}, sample=s, quality=quality)


def run_ref_cli(argv, cwd):
    r = subprocess.run([sys.executable, os.path.join(REF, "wisecondor.py")] + argv, cwd=cwd, capture_output=True,
                       text=True)
    if r.returncode != 0:
        raise RuntimeError("reference CLI failed: %s\n%s\n%s" % (argv, r.stdout[-2000:], r.stderr[-2000:]))
    return r.stdout


def tiny_counts():
    """Reference set (24 samples) and test samples (clean, gain, loss, spike + short run) of the tiny genome."""
    bins, lam, fac = synth.bin_model(TINY_BINSIZE, bin_seed=1, scale_bins=TINY_BINS, zero_frac=0.05)
    ref = synth.sample_counts(24, lam, fac, seed=2)
    tests = synth.sample_counts(4, lam, fac, seed=3)
    synth.inject_aberration(tests[1], bins, 3, 0.2, 0.7, 1.3, seed=4)        # long gain on chr3
    synth.inject_aberration(tests[2], bins, 7, 0.0, 1.0, 0.8, seed=5)        # whole-chromosome loss on chr7
    synth.inject_aberration(tests[3], bins, 1, 0.5, 0.52, 2.0, seed=6)       # single-bin spike on chr1
    synth.inject_aberration(tests[3], bins, 12, 0.3, 0.5, 0.6, seed=7)       # short deletion on chr12
    return bins, ref, tests


def golden_cli_tiny():
    """newref + test through the reference CLI; stores the reference npz arrays, the prep arrays that pin PCA,
    and one result set per test sample."""
    bins, ref, tests = tiny_counts()
    tmp = tempfile.mkdtemp(prefix="wc_golden_")
    try:
        names = []
        for i in range(ref.shape[0]):
            names.append("r%02d.npz" % i)
            write_sample_npz(os.path.join(tmp, names[-1]), ref[i], bins, TINY_BINSIZE)
        # keep the prep file: run the three cluster-mode steps (wisecondor.py:393-439) = newref without clean-up
        run_ref_cli(["newrefprep"] + names + ["ref_prep.npz"], tmp)
        for part in (1, 2, 3):
            run_ref_cli(["newrefpart", "ref_prep.npz", "ref_part", str(part), "3", "-refsize", "40"], tmp)
        run_ref_cli(["newrefpost", "ref_prep.npz", "ref_part", "3", "ref.npz"], tmp)
        prep = np.load(os.path.join(tmp, "ref_prep.npz"), allow_pickle=True)
        refnpz = np.load(os.path.join(tmp, "ref.npz"), allow_pickle=True)
        out = dict(
            bins=np.array(bins), binsize=TINY_BINSIZE, ref_counts=ref, test_counts=tests,
            prep_mask=prep['mask'], prep_maskedChromBins=prep['maskedChromBins'],
            prep_maskedChromBinSums=prep['maskedChromBinSums'], prep_correctedData=np.ascontiguousarray(prep['correctedData']),
            prep_maskedData=np.ascontiguousarray(prep['maskedData']),
            ref_binsize=refnpz['binsize'], ref_indexes=refnpz['indexes'], ref_distances=refnpz['distances'],
            ref_chromosome_sizes=refnpz['chromosome_sizes'], ref_mask=refnpz['mask'],
            ref_masked_sizes=refnpz['masked_sizes'], ref_pca_components=refnpz['pca_components'],
            ref_pca_mean=refnpz['pca_mean'])
        for t in range(tests.shape[0]):
            write_sample_npz(os.path.join(tmp, "t%d.npz" % t), tests[t], bins, TINY_BINSIZE)
            extra = ["-minrefbins", "10"] + (["-repeats", "3"] if t == 2 else [])
            run_ref_cli(["test", "t%d.npz" % t, "o%d.npz" % t, "ref.npz"] + extra, tmp)
            res = np.load(os.path.join(tmp, "o%d.npz" % t), allow_pickle=True)
            out["res%d_z" % t] = np.concatenate(list(res['results_z']))
            out["res%d_r" % t] = np.concatenate(list(res['results_r']))
            out["res%d_cwz" % t] = res['results_cwz']
            out["res%d_calls" % t] = np.asarray(res['results_calls'], dtype=float).reshape(-1, 5)
            out["res%d_scalars" % t] = np.array([res['threshold_z'], res['asdef'], res['aasdef']], dtype=float)
        np.savez_compressed(os.path.join(HERE, "tiny_cli.npz"), **out)
        print("tiny_cli.npz: N=%d masked, calls per test sample: %s" % (
            refnpz['indexes'].shape[0], [out["res%d_calls" % t].shape[0] for t in range(tests.shape[0])]))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def golden_functions():
    """Function-level vectors, produced by importing the reference's modules."""
    sys.path.insert(0, REF)
    with contextlib.redirect_stdout(io.StringIO()):
        import triarray as ref_tri    # noqa: F401
        import wisetools as ref_wt
    rng = np.random.default_rng(11)
    out = {}

    # ---- search: getReference on a 4-chromosome toy matrix, several part splits, ties and NaN ------------
    bins = [30, 22, 17, 9]
    n = sum(bins)
    X = 1.0 + rng.normal(0, 0.05, size=(n, 12))
    X[40] = X[3]                       # exact duplicate across chromosomes -> distance 0
    X[50] = X[60]                      # duplicate pair on chromosomes 2/3
    X[10, 4] = np.nan                  # NaN row: never selected, and selects nothing
    Xf = np.asfortranarray(X)          # the layout the reference's arrays have after the prep-npz round trip
    sums = list(np.cumsum(bins))
    with contextlib.redirect_stdout(io.StringIO()):
        idx, dst = ref_wt.getReference(Xf, bins, sums, 15, 1, 1)
        parts = [ref_wt.getReference(Xf, bins, sums, 15, p, 3) for p in (1, 2, 3)]
        idx_few, dst_few = ref_wt.getReference(Xf, bins, sums, 60, 1, 1)     # more slots than candidates for chr1
    assert np.array_equal(np.concatenate([p[0] for p in parts]), idx)
    out.update(search_bins=np.array(bins), search_X=X, search_idx=idx, search_dst=dst, search_idx_few=idx_few,
               search_dst_few=dst_few)

    # ---- ingest / PCA -----------------------------------------------------------------------------------
    sbins, lam, fac = synth.bin_model(TINY_BINSIZE, bin_seed=5, scale_bins=[12, 9, 7] + [3] * 19, zero_frac=0.1)
    counts = synth.sample_counts(10, lam, fac, seed=6)
    samples = [synth.counts_to_sample_dict(counts[i], sbins, 50000000) for i in range(10)]
    with contextlib.redirect_stdout(io.StringIO()):
        masked, chrom_bins, mask = ref_wt.toNumpyArray(samples)
        corrected, pca = ref_wt.trainPCA(masked)
        scaled = ref_wt.scaleSample(samples[0], 1, 3)
        tvec = ref_wt.toNumpyRefFormat(samples[1], [b + (1 if i % 2 else -1) for i, b in enumerate(chrom_bins)],
                                       np.ones(sum(b + (1 if i % 2 else -1) for i, b in enumerate(chrom_bins)), dtype=bool))
        tref = ref_wt.toNumpyRefFormat(samples[2], chrom_bins, mask)
        applied = ref_wt.applyPCA(tref, pca.mean_, pca.components_)
    out.update(ingest_bins=np.array(sbins), ingest_counts=counts, ingest_masked=masked, ingest_mask=mask,
               ingest_corrected=np.ascontiguousarray(corrected), ingest_components=pca.components_,
               ingest_mean=pca.mean_, ingest_scaled_chr1=scaled['1'], ingest_scaled_chr2=scaled['2'],
               ingest_padtrunc=tvec, ingest_tref=tref, ingest_applied=applied)

    # ---- z-scores: trySample / repeatTest / getOptimalCutoff on the search toy ---------------------------
    X2 = 1.0 + rng.normal(0, 0.05, size=(n, 12))
    with contextlib.redirect_stdout(io.StringIO()):
        idx2, dst2 = ref_wt.getReference(np.asfortranarray(X2), bins, sums, 12, 1, 1)
    cutoff, _ = ref_wt.getOptimalCutoff(dst2, 3)
    test = 1.0 + rng.normal(0, 0.03, size=n)
    test[35:45] *= 1.25                       # an aberration that gets marked and removed from the references
    test[70] = 0.0
    with contextlib.redirect_stdout(io.StringIO()):
        z1, r1, s1, sd1 = ref_wt.trySample(test, np.copy(test), idx2, dst2, bins, sums, cutoff)
        z5, r5, s5, sd5 = ref_wt.repeatTest(np.copy(test), idx2, dst2, bins, sums, cutoff, 3.0, 5)
    out.update(z_bins=np.array(bins), z_idx=idx2, z_dst=dst2, z_cutoff=cutoff, z_test=test, z_pass1=np.array([z1, r1, s1]),
               z_pass1_sd=sd1, z_pass5=np.array([z5, r5, s5]), z_pass5_sd=sd5)

    # ---- segmentation: fillTri/fillTriMin + segmentTri -------------------------------------------------
    regions, results = [], []
    specs = [(40, []), (90, [(20, 45, 1.2)]), (150, [(10, 30, -1.0), (100, 140, 0.9)]), (7, [(0, 7, 3.0)]),
             (3, [(0, 3, -4.0)]), (1, [(0, 1, 9.0)]), (200, [(0, 200, 0.6)]), (64, [(30, 31, 8.0)]),
             (120, [(0, 5, 2.5), (110, 120, -2.5)]), (310, [(50, 260, 0.5), (270, 300, -1.5)])]
    for length, runs in specs:
        zreg = rng.normal(0, 1, size=length)
        for a, b, shift in runs:
            zreg[a:b] += shift
        tri = ref_wt.fillTri(zreg)
        segs = tri.segmentTri(3.5, 3)
        regions.append(zreg)
        results.append((tri.getValue(0, length - 1), segs))
    out['seg_n'] = np.array([len(r) for r in regions])
    out['seg_z'] = np.concatenate(regions)
    out['seg_cw'] = np.array([r[0] for r in results])
    out['seg_calls'] = np.array([[i, s[1][0], s[1][1], s[0]] for i, r in enumerate(results) for s in r[1]], dtype=float)
    # equal values: first-occurrence tie breaking (triarray.py:62-66)
    flat = np.full(25, 2.0)
    tri = ref_wt.fillTri(flat)
    out['seg_flat_calls'] = np.array([[s[1][0], s[1][1], s[0]] for s in tri.segmentTri(3.5, 3)], dtype=float)
    # fillTriMin with an effect-size filter (wisetools.py:475-487)
    zreg = rng.normal(0, 1, size=60)
    zreg[20:40] += 2.0
    rreg = 1.0 + rng.normal(0, 0.01, size=60)
    rreg[20:40] += 0.08
    tri = ref_wt.fillTriMin(zreg, rreg, 0.05)
    out.update(segmin_z=zreg, segmin_r=rreg, segmin_cw=tri.getValue(0, 59),
               segmin_calls=np.array([[s[1][0], s[1][1], s[0]] for s in tri.segmentTri(3.5, 3)], dtype=float))
    np.savez_compressed(os.path.join(HERE, "functions.npz"), **out)
    print("functions.npz: %d arrays, %d segmentation calls" % (len(out), out['seg_calls'].shape[0]))


def report_files(tmp):
    """A sample npz with the read counts `convert` stores and a result npz with the keys `test` writes (wisecondor.py:273-281)
    that `report` reads; calls with effect sizes on both sides of the default -mineffect 1.5.  Shared with the CPU test."""
    bins = TINY_BINS
    rng = np.random.default_rng(41)
    row = rng.integers(50, 400, size=sum(bins))
    write_sample_npz(os.path.join(tmp, "s.npz"), row, bins, TINY_BINSIZE)
    s = dict(np.load(os.path.join(tmp, "s.npz"), allow_pickle=True))
    quality = {'mapped': 9123456, 'unmapped': 23456, 'no_coordinate': 1200, 'filter_rmdup': 345678, 'filter_mapq': 456789,
               'pre_retro': 8400000, 'post_retro': 8312345, 'pair_fail': 77}
    np.savez_compressed(os.path.join(tmp, "s.npz"), arguments={'binsize': 1000000.0, 'retdist': 4, 'retthres': 4, 'infile': 'a.bam'},
                        runtime={}, sample=s['sample'].item(), quality=quality)
    calls = [[3, 10, 29, 7.123456, 0.0312], [7, 0, 39, -12.5, -0.0849], [1, 30, 30, 5.9, 0.004], [12, 4, 9, -6.25, -0.015001],
             [20, 2, 3, 6.0, 0.015]]
    np.savez_compressed(os.path.join(tmp, "o.npz"), binsize=TINY_BINSIZE, threshold_z=5.2345, asdef=0.04567, aasdef=0.0512349,
                        arguments={'minzscore': None, 'repeats': 5, 'minrefbins': 25, 'mineffectsize': 0.0},
                        runtime={}, results_calls=np.array(calls, dtype=object))


def golden_report():
    """The reference's `report` on report_files(), default and explicit -mineffect."""
    tmp = tempfile.mkdtemp(prefix="wc_golden_")
    try:
        report_files(tmp)
        out = {}
        for name, extra in (("default", []), ("mineffect0", ["-mineffect", "0"]), ("mineffect5", ["-mineffect", "5"])):
            out[name] = run_ref_cli(["report", "s.npz", "o.npz"] + extra, tmp)
        with open(os.path.join(HERE, "report.json"), "w") as f:
            json.dump(out, f, indent=1, sort_keys=True)
        print("report.json: %d variants, %d lines each at most" % (len(out), max(len(v.splitlines()) for v in out.values())))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def segmin_nonfinite_cases():
    """(name, z, r) regions with inf / NaN z-scores (reference sigma 0, wisetools.py:431) and inf / NaN ratios (reference
    mean 0) under the effect-size filter.  Shared with the tests."""
    rng = np.random.default_rng(77)
    cases = []

    def base(n=72):
        z = rng.normal(0, 1, size=n)
        r = 1.0 + rng.normal(0, 0.01, size=n)
        z[20:40] += 2.0
        r[20:40] += 0.08
        return z, r

    z, r = base(); z[25] = np.inf; cases.append(("posinf_inside", z, r))
    z, r = base(); z[30] = -np.inf; cases.append(("neginf_inside", z, r))
    z, r = base(); z[50] = np.nan; cases.append(("nan_outside", z, r))
    z, r = base(); z[30] = -np.inf; z[55] = np.inf; cases.append(("both_signs", z, r))
    z, r = base(); z[8] = np.nan; r[8] = np.nan; cases.append(("nan_ratio", z, r))
    z, r = base(); z[28] = np.inf; r[28] = np.inf; z[60] = np.nan; r[60] = np.nan; cases.append(("inf_ratio", z, r))
    z, r = base(); z[66] = np.inf; cases.append(("posinf_never_passes", z, r))
    z, r = base(); z[22] = np.nan; z[23] = np.inf; z[45] = -np.inf; r[44:48] -= 0.09; cases.append(("many", z, r))
    z, r = base(); r[3] = np.nan; r[35] = np.nan; cases.append(("nan_ratio_finite_z", z, r))
    return cases


def golden_segmin_nonfinite():
    """fillTriMin + segmentTri of the reference on segmin_nonfinite_cases() (np.seterr('ignore') as wisecondor.py sets)."""
    sys.path.insert(0, REF)
    with contextlib.redirect_stdout(io.StringIO()):
        import wisetools as ref_wt
    out = {}
    with np.errstate(all='ignore'), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for name, z, r in segmin_nonfinite_cases():
            tri = ref_wt.fillTriMin(z, r, 0.05)
            segs = tri.segmentTri(3.5, 3)
            out[name + "_cw"] = tri.getValue(0, len(z) - 1)
            out[name + "_calls"] = np.array([[s[1][0], s[1][1], s[0]] for s in segs], dtype=float).reshape(-1, 3)
            print(name, len(segs), [(s[1], float(s[0])) for s in segs][:6])
    np.savez_compressed(os.path.join(HERE, "segmin_nonfinite.npz"), **out)


def search_case(seed):
    """(bins, X, k) of tests/test_oracle_vs_ref.py::test_search_random: 2-6 chromosomes of 1-24 bins, 1-39 samples, k up
    to 29 (often more than a chromosome's candidates) and one duplicated row."""
    rng = np.random.default_rng(seed)
    bins = [int(b) for b in rng.integers(1, 25, size=int(rng.integers(2, 7)))]
    n, S, k = sum(bins), int(rng.integers(1, 40)), int(rng.integers(1, 30))
    X = 1.0 + rng.normal(0, 0.05, size=(n, S))
    X[rng.integers(0, n)] = X[rng.integers(0, n)]
    return bins, X, k


def zscore_case(seed):
    """(bins, X, test) of test_zscores_random; the search table is wc_oracle.get_reference(X, bins, sums, 9, 1, 1)."""
    rng = np.random.default_rng(100 + seed)
    bins = [int(b) for b in rng.integers(5, 30, size=4)]
    n = sum(bins)
    X = 1.0 + rng.normal(0, 0.05, size=(n, 10))
    test = 1.0 + rng.normal(0, 0.03, size=n)
    test[3:9] *= 1.3
    return bins, X, test


def segmentation_case(seed):
    """z of test_segmentation_random: 1-159 bins, one shifted run when there are more than 20."""
    rng = np.random.default_rng(200 + seed)
    n = int(rng.integers(1, 160))
    z = rng.normal(0, 1, size=n)
    if n > 20:
        a = int(rng.integers(0, n - 10))
        z[a:a + int(rng.integers(2, 10))] += rng.choice([-2.0, 2.0])
    return z


RANDOM_SEEDS = {"search": range(4), "zscores": range(3), "segmentation": range(4)}


def reference_random_outputs(ref_wt):
    """The reference's outputs on the seeded cases above: getReference, getOptimalCutoff + repeatTest(2.5, 4) on the
    oracle's table, fillTri + segmentTri(3.0, 3).  `ref_wt` is the reference's wisetools module."""
    import wc_oracle
    out = {}
    for seed in RANDOM_SEEDS["search"]:
        bins, X, k = search_case(seed)
        with contextlib.redirect_stdout(io.StringIO()):
            out["search%d_idx" % seed], out["search%d_dst" % seed] = ref_wt.getReference(
                np.asfortranarray(X), bins, list(np.cumsum(bins)), k, 1, 1)
    for seed in RANDOM_SEEDS["zscores"]:
        bins, X, test = zscore_case(seed)
        sums = list(np.cumsum(bins))
        idx, dst = wc_oracle.get_reference(X, bins, sums, 9, 1, 1)
        cutoff, _ = ref_wt.getOptimalCutoff(dst, 3)
        with contextlib.redirect_stdout(io.StringIO()):
            z, r, sizes, sd = ref_wt.repeatTest(np.copy(test), idx, dst, bins, sums, cutoff, 2.5, 4)
        out.update({"zscores%d_cutoff" % seed: cutoff, "zscores%d_z" % seed: z, "zscores%d_r" % seed: r,
                    "zscores%d_sizes" % seed: sizes, "zscores%d_sd" % seed: sd})
    for seed in RANDOM_SEEDS["segmentation"]:
        z = segmentation_case(seed)
        tri = ref_wt.fillTri(z)
        out["segmentation%d_cw" % seed] = tri.getValue(0, len(z) - 1)
        out["segmentation%d_calls" % seed] = np.array([[x, y, v] for v, (x, y) in tri.segmentTri(3.0, 3)],
                                                      dtype=float).reshape(-1, 3)
    return out


def golden_oracle_random():
    """reference_random_outputs of the reference itself, for tests/test_oracle_vs_ref.py where oracle/_ref is absent."""
    sys.path.insert(0, REF)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    with contextlib.redirect_stdout(io.StringIO()):
        import wisetools as ref_wt
    out = reference_random_outputs(ref_wt)
    np.savez_compressed(os.path.join(HERE, "oracle_random.npz"), **out)
    print("oracle_random.npz: %d arrays" % len(out))


def golden_cli_tiny_mineff():
    """The reference's `test -mineffectsize` (wisecondor.py:460, fillTriMin) on the tiny genome's test samples against the
    reference npz of tiny_cli.npz (rebuilt from its arrays, as tests/test_cli_gpu.py does): 0.25 keeps the 1.3x gain of
    sample 1 and zeroes the 0.8x loss of sample 2."""
    tiny = np.load(os.path.join(HERE, "tiny_cli.npz"), allow_pickle=True)
    bins = [int(b) for b in tiny['bins']]
    tmp = tempfile.mkdtemp(prefix="wc_golden_")
    try:
        np.savez_compressed(os.path.join(tmp, "goldref.npz"), arguments={}, runtime={}, binsize=tiny['ref_binsize'],
                            indexes=tiny['ref_indexes'], distances=tiny['ref_distances'],
                            chromosome_sizes=tiny['ref_chromosome_sizes'], mask=tiny['ref_mask'],
                            masked_sizes=tiny['ref_masked_sizes'], pca_components=tiny['ref_pca_components'],
                            pca_mean=tiny['ref_pca_mean'])
        out = {'mineffectsize': 0.25}
        for t in range(tiny['test_counts'].shape[0]):
            write_sample_npz(os.path.join(tmp, "t%d.npz" % t), tiny['test_counts'][t], bins, TINY_BINSIZE)
            run_ref_cli(["test", "t%d.npz" % t, "o%d.npz" % t, "goldref.npz", "-minrefbins", "10", "-mineffectsize", "0.25"], tmp)
            res = np.load(os.path.join(tmp, "o%d.npz" % t), allow_pickle=True)
            out["res%d_cwz" % t] = res['results_cwz']
            out["res%d_calls" % t] = np.asarray(res['results_calls'], dtype=float).reshape(-1, 5)
            out["res%d_z" % t] = np.concatenate(list(res['results_z']))
        np.savez_compressed(os.path.join(HERE, "tiny_cli_mineff.npz"), **out)
        print("tiny_cli_mineff.npz: calls per test sample with / without the filter: %s / %s" % (
            [out["res%d_calls" % t].shape[0] for t in range(4)], [tiny["res%d_calls" % t].shape[0] for t in range(4)]))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


FLAG_VARIANTS = [                                   # (name, test sample, sample bin size, extra flags of `test`)
    ("chromosomes", 1, None, ["-chromosomes", "1,3,7,12", "-minzscore", "4.0"]),
    ("multitest", 3, None, ["-multitest", "5"]),
    ("minzscore_repeats1", 2, None, ["-minzscore", "3.2", "-repeats", "1"]),
    ("rescaled_sample", 1, 500000, []),             # sample binned at 0.5 Mb: scaleSample sums pairs of bins (wisetools.py:20-44)
]


def split_counts(row, bins):
    """A 0.5 Mb sample whose pairs of bins sum to the 1 Mb counts (an odd split, so both halves matter)."""
    out, nb = [], []
    pos = 0
    for n in bins:
        c = row[pos:pos + n].astype(np.int64)
        fine = np.empty(2 * n, dtype=np.int64)
        fine[0::2] = c // 3
        fine[1::2] = c - c // 3
        out.append(fine)
        nb.append(2 * n)
        pos += n
    return np.concatenate(out), nb


def golden_cli_tiny_flags():
    """The reference's `test` with its remaining flags and with a sample of another bin size, same files as
    golden_cli_tiny_mineff."""
    tiny = np.load(os.path.join(HERE, "tiny_cli.npz"), allow_pickle=True)
    bins = [int(b) for b in tiny['bins']]
    tmp = tempfile.mkdtemp(prefix="wc_golden_")
    try:
        np.savez_compressed(os.path.join(tmp, "goldref.npz"), arguments={}, runtime={}, binsize=tiny['ref_binsize'],
                            indexes=tiny['ref_indexes'], distances=tiny['ref_distances'],
                            chromosome_sizes=tiny['ref_chromosome_sizes'], mask=tiny['ref_mask'],
                            masked_sizes=tiny['ref_masked_sizes'], pca_components=tiny['ref_pca_components'],
                            pca_mean=tiny['ref_pca_mean'])
        out = {}
        for name, t, sample_binsize, extra in FLAG_VARIANTS:
            if sample_binsize is None:
                write_sample_npz(os.path.join(tmp, name + ".npz"), tiny['test_counts'][t], bins, TINY_BINSIZE)
            else:
                fine, nb = split_counts(tiny['test_counts'][t], bins)
                write_sample_npz(os.path.join(tmp, name + ".npz"), fine, nb, sample_binsize)
            run_ref_cli(["test", name + ".npz", name + "_o.npz", "goldref.npz", "-minrefbins", "10"] + extra, tmp)
            res = np.load(os.path.join(tmp, name + "_o.npz"), allow_pickle=True)
            out[name + "_cwz"] = np.asarray(res['results_cwz'], dtype=float)
            out[name + "_calls"] = np.asarray(res['results_calls'], dtype=float).reshape(-1, 5)
            out[name + "_z"] = np.concatenate(list(res['results_z']))
            out[name + "_scalars"] = np.array([res['threshold_z'], res['asdef'], res['aasdef']], dtype=float)
            print(name, "calls", out[name + "_calls"].shape[0], "cwz", out[name + "_cwz"].shape, "threshold", float(res['threshold_z']))
        np.savez_compressed(os.path.join(HERE, "tiny_cli_flags.npz"), **out)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def golden_cli_tiny_prep_binsize():
    """The reference's `newrefprep -binsize 2000000` on the tiny genome's 1 Mb reference samples (every sample rescaled by
    scaleSample before the mask / PCA, wisecondor.py:99-101)."""
    tiny = np.load(os.path.join(HERE, "tiny_cli.npz"), allow_pickle=True)
    bins = [int(b) for b in tiny['bins']]
    tmp = tempfile.mkdtemp(prefix="wc_golden_")
    try:
        names = []
        for i in range(tiny['ref_counts'].shape[0]):
            names.append("r%02d.npz" % i)
            write_sample_npz(os.path.join(tmp, names[-1]), tiny['ref_counts'][i], bins, TINY_BINSIZE)
        run_ref_cli(["newrefprep"] + names + ["prep2.npz", "-binsize", "2000000"], tmp)
        prep = np.load(os.path.join(tmp, "prep2.npz"), allow_pickle=True)
        np.savez_compressed(os.path.join(HERE, "tiny_cli_prep_binsize.npz"), binsize=prep['binsize'], mask=prep['mask'],
                            chromosomeBins=prep['chromosomeBins'], maskedChromBins=prep['maskedChromBins'],
                            maskedChromBinSums=prep['maskedChromBinSums'], maskedData=np.ascontiguousarray(prep['maskedData']),
                            correctedData=np.ascontiguousarray(prep['correctedData']))
        print("tiny_cli_prep_binsize.npz: binsize", prep['binsize'], "bins", list(prep['chromosomeBins'])[:4], "masked", int(sum(prep['maskedChromBins'])))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    if not os.path.isfile(os.path.join(REF, "wisetools.py")):
        rc = subprocess.call([sys.executable, os.path.join(ROOT, "oracle", "make_ref.py")])
        if rc != 0:
            print("the reference is not available: golden vectors can only be regenerated in the build container")
            return 1
    if '--report-only' in sys.argv:
        golden_report()
        return 0
    if '--prep-binsize-only' in sys.argv:
        golden_cli_tiny_prep_binsize()
        return 0
    if '--flags-only' in sys.argv:
        golden_cli_tiny_flags()
        return 0
    if '--mineff-only' in sys.argv:
        golden_cli_tiny_mineff()
        return 0
    if '--segmin-only' in sys.argv:
        golden_segmin_nonfinite()
        return 0
    if '--random-only' in sys.argv:
        golden_oracle_random()
        return 0
    golden_functions()
    golden_cli_tiny()
    golden_report()
    golden_segmin_nonfinite()
    golden_cli_tiny_mineff()
    golden_cli_tiny_flags()
    golden_cli_tiny_prep_binsize()
    golden_oracle_random()
    return 0


if __name__ == "__main__":
    sys.exit(main())
