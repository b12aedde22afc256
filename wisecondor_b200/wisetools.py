"""Host-side mirror of the reference's numerics library (/root/reference/wisetools.py) for the hot path.

Same function names, argument meaning and return values as the reference; the bodies call the CUDA library
through wisecondor_b200._cabi / wisecondor_b200.device.  Functions the north star keeps on the host
(scaleSample, getOptimalCutoff, getPart, splitByChrom, inflateArray) are plain numpy.
"""
import time

import numpy as np

from . import _mem
from . import device as _dev

DEVICE = 0   # CUDA device the host-facing functions use


def getPart(partnum, outof, bincount):
    """Start and end bin of 0-based part `partnum` of `outof` (reference wisetools.py:358-361)."""
    return int(bincount / float(outof) * partnum), int(bincount / float(outof) * (partnum + 1))


def getReference(correctedData, chromosomeBins, chromosomeBinSums, selectRefAmount=100, part=1, splitParts=1,
                 device=None):
    """Reference bins for the rows of 1-based `part` of `splitParts` (reference wisetools.py:364-398).

    Returns (indexArray int32 rows x selectRefAmount, distanceArray float64 rows x selectRefAmount): per target
    bin the positions, within the concatenation of all other chromosomes, of the selectRefAmount nearest bins
    ordered by (squared distance, index), and those distances.  The chromosome split of the reference's
    splitByChrom/getRefForBins loop happens inside the kernel (per-row exclusion ranges).  correctedData may be a
    numpy array [N][S] or a device array; `device` overrides the module-level DEVICE (one host thread per GPU).
    """
    timeStart = time.time()
    bincount = int(chromosomeBinSums[-1])
    startNum, endNum = getPart(part - 1, splitParts, bincount)
    print('Working on part', part, 'of', splitParts, 'meaning bins', startNum, 'up to', endNum)
    dev = DEVICE if device is None else device
    bins = [int(b) for b in chromosomeBins]
    if _mem.is_device(correctedData):
        if correctedData.shape[0] != bincount:
            raise ValueError("correctedData has %d bins, chromosomeBinSums says %d" % (correctedData.shape[0], bincount))
        idx, dist = _dev.newref_search(correctedData, bins, startNum, endNum, int(selectRefAmount))
        idx, dist = _mem.to_host(idx), _mem.to_host(dist)
    else:
        X = np.ascontiguousarray(correctedData, dtype=np.float64)
        if X.shape[0] != bincount:
            raise ValueError("correctedData has %d bins, chromosomeBinSums says %d" % (X.shape[0], bincount))
        idx, dist = _dev.newref_search(X, bins, startNum, endNum, int(selectRefAmount), device=dev)
    print('Time spent:', int(time.time() - timeStart), 'seconds')
    return idx, dist


class _FittedPCA(object):
    """What the reference reads from the scikit-learn object trainPCA returns (wisecondor.py:107-108)."""

    def __init__(self, components, mean):
        self.components_ = components
        self.mean_ = mean
        self.n_components_ = components.shape[0]


def _stackCounts(samples):
    """Host part of toNumpyArray (reference wisetools.py:244-253): chromosomes 1..22 of every sample, stacked
    sample-major [S][Nraw] int32.  Like the reference, samples whose chromosome lengths differ are an error."""
    chromBins = []
    for chromosome in range(1, 23):
        lens = set(int(np.asarray(s[str(chromosome)]).shape[0]) for s in samples)
        if len(lens) != 1:
            raise ValueError("could not broadcast: chromosome %d has differing bin counts %s" % (chromosome, sorted(lens)))
        chromBins.append(lens.pop())
    counts = np.empty((len(samples), sum(chromBins)), dtype=np.int32)
    for i, s in enumerate(samples):
        counts[i] = np.concatenate([np.asarray(s[str(c)]) for c in range(1, 23)])
    return counts, chromBins


def toNumpyArray(samples, as_device=False):
    """reference wisetools.py:240-264.  Returns (maskedData [N][S], chromBins, mask)."""
    counts, chromBins = _stackCounts(samples)
    masked, mask = _dev.newref_normalize(_mem.to_device(counts, DEVICE))
    print('Applying nonzero mask on the data:', (counts.shape[1], counts.shape[0]), 'becomes', tuple(masked.shape))
    return (masked if as_device else _mem.to_host(masked)), chromBins, mask


def trainPCA(refData, pcacomp=3, as_device=False):
    """reference wisetools.py:89-101.  refData: [N][S] numpy or device array.  Returns (corrected [N][S], pca) where
    pca carries components_ and mean_."""
    X = refData if _mem.is_device(refData) else _mem.to_device(np.ascontiguousarray(refData, dtype=np.float64), DEVICE)
    corrected, comps, mean = _dev.pca_fit_apply(X, pcacomp)
    return (corrected if as_device else _mem.to_host(corrected)), _FittedPCA(comps, mean)


def getOptimalCutoff(reference, repeats):
    """mean + 3 sigma of the distances below the previous cutoff, `repeats` rounds (reference
    wisetools.py:328-336).  Sample independent, computed once per reference on the host with numpy so the
    value is bit-identical to the reference's."""
    optimalCutoff = float("inf")
    mask = np.zeros(reference.shape)
    for _ in range(repeats):
        mask = reference < optimalCutoff
        optimalCutoff = np.average(reference[mask]) + 3 * np.std(reference[mask])
    return optimalCutoff, mask


def scaleSample(sample, fromSize, toSize):
    """Down-bin a sample dict by an integer factor (reference wisetools.py:220-237).  Host."""
    if fromSize == toSize or toSize is None:
        return sample
    if toSize == 0 or fromSize == 0 or toSize < fromSize or toSize % fromSize > 0:
        print('ERROR: Impossible binsize scaling requested:', fromSize, 'to', toSize)
        raise SystemExit(1)
    scale = int(toSize // fromSize)
    out = dict()
    for chrom in sample:
        data = np.asarray(sample[chrom])
        newLen = int(np.ceil(len(data) / float(scale)))
        padded = np.zeros(newLen * scale, dtype=np.int64)
        padded[:len(data)] = data
        out[chrom] = padded.reshape(newLen, scale).sum(axis=1).astype(np.int32)
    return out


def inflateArray(array, mask):
    """Scatter `array` into the True positions of `mask`, zeros elsewhere (reference wisetools.py:281-288)."""
    temp = np.zeros(mask.shape[0])
    temp[np.asarray(mask, dtype=bool)] = array
    return temp


def inflateArrayMulti(array, mask_list):
    """reference wisetools.py:291-295."""
    temp = array
    for mask in reversed(mask_list):
        temp = inflateArray(temp, mask)
    return temp


# ------------------------------------------------------------------------------------------------------------
# test path
# ------------------------------------------------------------------------------------------------------------
def _f64(array):
    return _mem.to_device(np.ascontiguousarray(array, dtype=np.float64), DEVICE)


def _refFormatCounts(sample, chromBins):
    """Host part of toNumpyRefFormat (reference wisetools.py:268-273): per autosome zero-pad / truncate the
    count array to chromBins[c] and concatenate.  Returns int32 [Nraw]."""
    parts = []
    for chromosome in range(1, 23):
        want = int(chromBins[chromosome - 1])
        have = np.asarray(sample[str(chromosome)])
        thisChrom = np.zeros(want, dtype=np.int32)
        minLen = min(want, len(have))
        thisChrom[:minLen] = have[:minLen]
        parts.append(thisChrom)
    return np.concatenate(parts)


def toNumpyRefFormat(sample, chromBins, mask):
    """reference wisetools.py:267-278: masked, total-normalised bin vector of one sample (numpy float64 [N])."""
    return prepSamples([sample], chromBins, mask, None, None)[:, 0].copy()


def applyPCA(sampleData, mean, components):
    """reference wisetools.py:104-113: sampleData / ((sampleData - mean) C^T C + mean)."""
    out = _dev.apply_pca(_f64(np.asarray(sampleData, dtype=np.float64)[None, :]), _f64(mean), _f64(components))
    return _mem.to_host(out)[:, 0].copy()


def prepSample(sample, chromosome_sizes, mask, pca_mean, pca_components):
    """reference wisetools.py:401-404."""
    return prepSamples([sample], chromosome_sizes, mask, pca_mean, pca_components)[:, 0].copy()


def prepSamples(samples, chromosome_sizes, mask, pca_mean, pca_components, as_device=False):
    """prepSample for a batch: returns T [N][B'] (bin-major, sample-minor; B' = B rounded up to 32 when
    as_device, else exactly B as numpy)."""
    counts = np.stack([_refFormatCounts(s, chromosome_sizes) for s in samples])
    masked_raw = np.flatnonzero(np.asarray(mask, dtype=bool)).astype(np.int32)
    pm = pc = None
    if pca_components is not None:
        pm, pc = _f64(pca_mean), _f64(pca_components)
    T = _dev.test_prep(_mem.to_device(counts, DEVICE), _mem.to_device(masked_raw, DEVICE), pm, pc)
    if as_device:
        return T
    return _mem.to_host(T)[:, :len(samples)]


_TABLE_CACHE = {}


def _table(indexes, distances, chromosomeBins, cutoff):
    key = (id(indexes), id(distances), float(cutoff), DEVICE)
    hit = _TABLE_CACHE.get(key)
    if hit is None or hit[0] is not indexes:
        _TABLE_CACHE.clear()
        hit = (indexes, _dev.ReferenceTable(indexes, distances, chromosomeBins, cutoff, device=DEVICE))
        _TABLE_CACHE[key] = hit
    return hit[1]


def repeatTestBatch(testData, indexes, distances, chromosomeBins, chromosomeBinSums, cutoff, threshold, repeats):
    """repeatTest for many samples at once.  testData: numpy [B][N] (one corrected sample per row).
    Returns (resultsZ [B][N], resultsR [B][N], refSizes [B][N] float, stdDevAvg [B])."""
    X = np.asarray(testData, dtype=np.float64)
    b, n = X.shape
    T = np.ones((n, _dev.pad32(b)))                      # bin-major, sample-minor, padded to whole warps of samples
    T[:, :b] = X.T
    table = _table(indexes, distances, chromosomeBins, cutoff)
    z, r, sizes, asdef = _dev.zscore_batch(_f64(T), b, table, threshold, repeats)
    return _mem.to_host(z), _mem.to_host(r), _mem.to_host(sizes).astype(float), _mem.to_host(asdef)


def trySample(testData, testCopy, indexes, distances, chromosomeBins, chromosomeBinSums, cutoff):
    """reference wisetools.py:407-435: one z-score pass.  `testCopy` carries the -1 marks of earlier passes."""
    n = len(testData)
    T = np.ones((n, 32))
    C = np.ones((n, 32))
    T[:, 0] = np.asarray(testData, dtype=np.float64)
    C[:, 0] = np.asarray(testCopy, dtype=np.float64)
    table = _table(indexes, distances, chromosomeBins, cutoff)
    z, r, sizes, asdef = _dev.zscore_batch(_f64(T), 1, table, float("inf"), 1, copy_init=_f64(C))
    return _mem.to_host(z)[0], _mem.to_host(r)[0], _mem.to_host(sizes)[0].astype(float), float(_mem.to_host(asdef)[0])


def repeatTest(testData, indexes, distances, chromosomeBins, chromosomeBinSums, cutoff, threshold, repeats):
    """reference wisetools.py:438-448 for one sample."""
    z, r, sizes, asdef = repeatTestBatch(np.asarray(testData)[None, :], indexes, distances, chromosomeBins,
                                         chromosomeBinSums, cutoff, threshold, repeats)
    return z[0], r[0], sizes[0], float(asdef[0])


def segmentChromosomes(cleanedZ_or_z, refSizes, masked_sizes, chromosomes, minrefbins, z_threshold, min_search=3,
                       resultsR=None, mineffectsize=0):
    """fillTriMin + segmentTri for the listed chromosomes (1-based, as -chromosomes) of a batch (reference
    wisecondor.py:233-238, wisetools.py:466-487, triarray.py:59-84).  z, refSizes (and resultsR when
    mineffectsize != 0): numpy [B][N].
    Returns (chromWide [B][nsel], cleanedBins [B][nsel], calls structured array sorted by (sample, chrom, x))."""
    z = _f64(cleanedZ_or_z)
    sizes = _mem.to_device(np.ascontiguousarray(refSizes).astype(np.int32), DEVICE)
    r = None
    if mineffectsize != 0:
        r = _f64(resultsR)
    cwz, cleaned, calls = _dev.segment_batch(z, sizes, masked_sizes, [c - 1 for c in chromosomes], minrefbins,
                                             z_threshold, min_search, r=r, mineffectsize=mineffectsize)
    return _mem.to_host(cwz), _mem.to_host(cleaned), calls


def testSamples(samples, ref, z_threshold, chromosomes=tuple(range(1, 23)), mineffectsize=0, minrefbins=25, repeats=5,
                min_search=3, batch=1024):
    """The computation of toolTest (reference wisecondor.py:196-268) for a list of sample dicts already scaled to
    the reference's binsize.  `ref` holds the reference-npz entries.  Returns one dict per sample with the
    result-npz entries results_r, results_z, results_cwz, results_calls, threshold_z, asdef, aasdef.

    Device: prepSample (K7), repeatTest (K8), fillTriMin + segmentTri (K9).  Host: getOptimalCutoff (once per
    reference), the cleaned->raw coordinate walk and the per-call median of R (wisecondor.py:241-257), inflate."""
    chromosome_sizes = [int(v) for v in ref['chromosome_sizes']]
    masked_sizes = [int(v) for v in ref['masked_sizes']]
    mask = np.asarray(ref['mask'], dtype=bool)
    optimalCutoff, _ = getOptimalCutoff(ref['distances'], 3)
    table = _table(ref['indexes'], ref['distances'], masked_sizes, optimalCutoff)
    masked_raw = np.flatnonzero(mask)
    raw_starts = np.concatenate(([0], np.cumsum(chromosome_sizes)))
    masked_starts = np.concatenate(([0], np.cumsum(masked_sizes)))
    sel = [c - 1 for c in chromosomes]
    out = []
    timeStartTest = time.time()
    native = _mem.BACKEND == "native"
    if not native:
        torch = _mem.torch()
        dev = torch.device("cuda", DEVICE)
        copy_stream = torch.cuda.Stream(device=dev)

    def assemble(pending):
        """Host glue of one finished chunk (wisecondor.py:214-222, 241-268): keep mask, cleaned->raw walk, medians, inflate."""
        nb, host, calls, done = pending
        if done is not None:
            done.synchronize()
        z_h, r_h, sizes_h, asdef_h, cwz_h = [t if isinstance(t, np.ndarray) else t.numpy() for t in host]
        call_lo = np.searchsorted(calls['sample'], np.arange(nb), side='left')
        call_hi = np.searchsorted(calls['sample'], np.arange(nb), side='right')
        for b in range(nb):
            keep = sizes_h[b] >= minrefbins                                  # infinite_mask, wisecondor.py:215
            cleanedR = r_h[b][keep]
            kept_raw = masked_raw[keep]                                      # raw bin of every cleaned bin
            kept_starts = np.searchsorted(kept_raw, raw_starts)              # cleaned offset of every chromosome
            inflatedZ = np.zeros(mask.shape[0])
            inflatedR = np.zeros(mask.shape[0])
            inflatedZ[kept_raw] = z_h[b][keep]
            inflatedR[kept_raw] = cleanedR - 1
            stouffCalls = []
            for c in calls[call_lo[b]:call_hi[b]]:
                chrom = sel[int(c['chrom'])]
                x, y = int(c['x']), int(c['y'])
                base = kept_starts[chrom]
                pos = kept_raw[base:kept_starts[chrom + 1]] - raw_starts[chrom]
                start_raw = int(pos[x])
                end_raw = int(pos[y - 1]) + 1 if y > x else start_raw        # the walk of wisecondor.py:242-253
                stouffCalls.append([chrom + 1, start_raw, end_raw, float(c['z']),
                                    np.median(cleanedR[base + x:base + y + 1]) - 1])
            asdef = float(asdef_h[b])
            out.append(dict(
                results_z=[inflatedZ[raw_starts[i]:raw_starts[i + 1]] for i in range(len(chromosome_sizes))],
                results_r=[inflatedR[raw_starts[i]:raw_starts[i + 1]] for i in range(len(chromosome_sizes))],
                results_cwz=cwz_h[b].copy(), results_calls=np.array(stouffCalls), threshold_z=z_threshold,
                asdef=asdef, aasdef=asdef * z_threshold))

    # Pipeline over chunks: the z-score kernels of chunk i run while the host assembles chunk i-1, and the results of
    # chunk i travel to (pinned) host memory on a second stream while chunk i+1 computes.
    pending = None
    for first in range(0, len(samples), batch):
        chunk = samples[first:first + batch]
        nb = len(chunk)
        T = prepSamples(chunk, chromosome_sizes, mask, ref['pca_mean'], ref['pca_components'], as_device=True)
        z_d, r_d, sizes_d, asdef_d = _dev.zscore_batch(T, nb, table, z_threshold, repeats)       # asynchronous
        if pending is not None:
            assemble(pending)
        cwz_d, cleaned_d, calls = _dev.segment_batch(z_d, sizes_d, masked_sizes, sel, minrefbins, z_threshold, min_search,
                                                     r=r_d if mineffectsize != 0 else None, mineffectsize=mineffectsize)
        if native:                                        # synchronous copies on the default stream
            pending = (nb, [_mem.to_host(t) for t in (z_d, r_d, sizes_d, asdef_d, cwz_d)], calls, None)
            continue
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream(dev))
        host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in (z_d, r_d, sizes_d, asdef_d, cwz_d)]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ready)
            for h, t in zip(host, (z_d, r_d, sizes_d, asdef_d, cwz_d)):
                h.copy_(t, non_blocking=True)
                t.record_stream(copy_stream)
            done = torch.cuda.Event()
            done.record(copy_stream)
        pending = (nb, host, calls, done)
    if pending is not None:
        assemble(pending)
    del masked_starts
    print('Time spent on obtaining z-scores and stouffers z-scores:', int(time.time() - timeStartTest), 'seconds')
    return out
