#!/usr/bin/env python
"""wisecondor.py - drop-in command line of WISECONDOR's within-sample comparison path on B200.

Same sub-commands, positional arguments, flags, defaults, intermediate file names and npz keys as the reference's
wisecondor.py (/root/reference/wisecondor.py:345-521), so scripts such as the reference's run.sh keep working:

    newref      infiles... outfile [-refsize 100 -binsize None -cpus 1 -parts 1] [-gpus N]
    newrefprep  infiles... prepfile [-binsize]
    newrefpart  prepfile partfile m n [-refsize 100]
    newrefpost  prepfile partfile parts outfile
    test        infile outfile reference [-minzscore -chromosomes -mineffectsize 0 -multitest 1000 -minrefbins 25 -repeats 5]
    testbatch   infiles... outdir reference [same flags as test]      (new: many samples per launch)

The arithmetic of every one of them runs in libwisecondor_b200.so (hand-written sm_100a kernels) through
wisecondor_b200.wisetools; there is no CPU fallback.  `report` (text formatting of a sample npz and a result npz) is
kept as a host tool.  `convert` and `plot` are host-only tools of the reference that this build does not replace (BAM
binning stays on the host with pysam; plotting only reads the result npz, whose keys are unchanged) - they are declared
so that the interface is complete and say so when used.

The tool functions keep the reference's names (toolNewref, toolTest, ...) because every npz stores
`arguments=vars(args)`, which pickles `args.func` by name (/root/reference/README.md:154).
"""
import argparse
import datetime
import getpass
import os
import socket
import subprocess
import sys
import threading
import time

import numpy as np

from wisecondor_b200 import _mem, wisetools

curTime = datetime.datetime.now()


# ---- runtime metadata stored in every npz (reference wisetools.py:47-70) -----------------------------------------
def getVersion():
    try:
        return subprocess.check_output(["git", "describe", "--always"], stderr=subprocess.DEVNULL).split()[0]
    except Exception:
        return 'unknown'


def getRuntime():
    return {'version': getVersion(), 'datetime': curTime, 'hostname': socket.gethostname(),
            'username': getpass.getuser(), 'backend': 'wisecondor_b200 (sm_100a)'}


def printArgs(args):
    argdict = vars(args)
    print('tool =', str(argdict['func']).split()[1][4:])
    for arg in sorted(argdict.keys()):
        if arg != 'func':
            print(arg, '=', argdict[arg])


def _load(path):
    return np.load(path, allow_pickle=True, encoding='latin1')


def _ragged(arrays):
    out = np.empty(len(arrays), dtype=object)
    for i, a in enumerate(arrays):
        out[i] = a
    return out


# ---- newref ---------------------------------------------------------------------------------------------------------
def toolNewref(args):
    """reference wisecondor.py:30-69: prep -> parts -> post, skipping files that already exist (resume)."""
    head, tail = os.path.split(args.outfile)
    if tail[-4:] == '.npz':
        tail = tail[:-4]
    basePath = os.path.join(head, tail)
    args.prepfile = basePath + "_prep.npz"
    args.partfile = basePath + "_part"
    gpus = max(1, int(getattr(args, 'gpus', 1) or 1))
    args.parts = max(args.parts, args.cpus, gpus)

    if not os.path.isfile(args.prepfile):
        toolNewrefPrep(args)

    todo = [p for p in range(1, args.parts + 1) if not os.path.isfile(args.partfile + "_" + str(p) + ".npz")]
    if gpus > 1 and len(todo) == args.parts and not getattr(args, 'partfiles', False):
        # The multi-GPU product path: one process per GPU, every rank searches its getPart rows of the whole matrix, the
        # rows travel over NCCL (all-gather) instead of part files (reference wisecondor.py:146-158) and rank 0 writes the
        # reference npz.  Resume granularity: the prep file.
        _spawnRanks(gpus, ['newrefrank', args.prepfile, args.outfile, '-refsize', str(args.refsize)])
        os.remove(args.prepfile)
        return
    if gpus > 1 and todo:
        # one host thread per GPU; the C ABI releases the GIL for the duration of each search
        import copy
        errors = []

        def worker(dev, parts):
            try:
                for part in parts:
                    thisArgs = copy.copy(args)
                    thisArgs.part = [part, args.parts]
                    toolNewrefPart(thisArgs, device=dev)
            except BaseException as exc:      # surfaced below: a failed part must not be silent
                errors.append(exc)

        threads = [threading.Thread(target=worker, args=(d, todo[d::gpus])) for d in range(gpus)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
    else:
        for part in todo:
            args.part = [part, args.parts]
            toolNewrefPart(args)

    toolNewrefPost(args)
    os.remove(args.prepfile)
    for part in range(1, args.parts + 1):
        os.remove(args.partfile + '_' + str(part) + '.npz')


def _spawnRanks(world, argv):
    """Run `wisecondor.py <argv>` once per GPU with the torch.distributed environment of a single-node job (what torchrun
    would set); any failing rank fails the command."""
    import socket as _socket
    with _socket.socket() as sock:
        sock.bind(('127.0.0.1', 0))
        port = sock.getsockname()[1]
    procs = []
    for rank in range(world):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR='127.0.0.1',
                   MASTER_PORT=str(port), WISECONDOR_BACKEND='torch')
        procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__)] + argv, env=env))
    codes = [p.wait() for p in procs]
    if any(codes):
        print('ERROR: rank exit codes', codes)
        sys.exit(1)


def toolNewrefRank(args):
    """One rank of `newref -gpus N` (internal sub-command, started by _spawnRanks): the reference's newrefpart for part
    RANK+1 of WORLD_SIZE (wisecondor.py:111-132) with NCCL instead of files - 1/N of the corrected matrix uploaded per rank
    and all-gathered over NVLink, the search of the rank's getPart rows, an all-gather of the (rows x refsize) blocks -
    then, on rank 0, newrefpost's writer (wisecondor.py:160-170)."""
    import torch
    import torch.distributed as dist
    from wisecondor_b200 import shard
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    npzdata = _load(args.prepfile)
    maskedChromBins = [int(v) for v in npzdata['maskedChromBins']]
    corrected = torch.from_numpy(np.ascontiguousarray(npzdata['correctedData'], dtype=np.float64)).pin_memory()
    n, s = corrected.shape
    timeStart = time.time()
    job = shard.ShardedSearch(n, s, args.refsize, rank, world, dev)
    job.run(corrected, maskedChromBins)
    idx, dst = shard.allgather_rows(job.idx, job.dist, n)
    torch.cuda.synchronize(dev)
    if rank == 0:
        print('Time spent on the search over', world, 'GPUs:', round(time.time() - timeStart, 3), 'seconds')
        np.savez_compressed(args.outfile,
                            arguments=vars(args),
                            runtime=getRuntime(),
                            binsize=npzdata['binsize'].item(),
                            indexes=idx.cpu().numpy(),
                            distances=dst.cpu().numpy(),
                            chromosome_sizes=npzdata['chromosomeBins'],
                            mask=npzdata['mask'],
                            masked_sizes=npzdata['maskedChromBins'],
                            pca_components=npzdata['pca_components'],
                            pca_mean=npzdata['pca_mean'])
    dist.barrier()
    dist.destroy_process_group()


def toolNewrefPrep(args):
    """reference wisecondor.py:72-108."""
    samples = []
    binsizes = set()
    for infile in args.infiles:
        print('Loading:', infile, end=" ")
        npzdata = _load(infile)
        sampleBinSize = npzdata['arguments'].item()['binsize']
        print(' \tbinsize:', int(sampleBinSize))
        samples.append(wisetools.scaleSample(npzdata['sample'].item(), sampleBinSize, args.binsize))
        binsizes.add(sampleBinSize)

    if args.binsize is None and len(binsizes) != 1:
        print('ERROR: There appears to be a mismatch in binsizes in your dataset:', binsizes)
        print('Either remove the offending sample or use -binsize to scale all samples')
        sys.exit(1)
    binsize = args.binsize
    if args.binsize is None:
        binsize = binsizes.pop()

    maskedData, chromosomeBins, mask = wisetools.toNumpyArray(samples, as_device=True)
    del samples
    starts = np.concatenate(([0], np.cumsum(chromosomeBins)))
    maskedChromBins = [int(np.sum(mask[starts[i]:starts[i + 1]])) for i in range(len(chromosomeBins))]
    maskedChromBinSums = [int(v) for v in np.cumsum(maskedChromBins)]
    correctedData, pca = wisetools.trainPCA(maskedData, as_device=True)
    np.savez_compressed(args.prepfile,
                        arguments=vars(args),
                        runtime=getRuntime(),
                        binsize=binsize,
                        chromosomeBins=chromosomeBins,
                        maskedData=_mem.to_host(maskedData),
                        mask=mask,
                        maskedChromBins=maskedChromBins,
                        maskedChromBinSums=maskedChromBinSums,
                        # Fortran order, like the transposed view the reference saves (wisetools.py:101): a reference CPU
                        # worker that reads this file then sums over samples in the same (sequential) order
                        correctedData=np.asfortranarray(_mem.to_host(correctedData)),
                        pca_components=pca.components_,
                        pca_mean=pca.mean_)


def toolNewrefPart(args, device=None):
    """reference wisecondor.py:111-132."""
    if args.part[0] > args.part[1]:
        print('ERROR: Part should be smaller or equal to total parts:', args.part[0], '>', args.part[1], 'is wrong')
        sys.exit(1)
    if args.part[0] < 0:
        print('ERROR: Part should be at least zero:', args.part[0], '<', 0, 'is wrong')
        sys.exit(1)

    npzdata = _load(args.prepfile)
    correctedData = npzdata['correctedData']
    maskedChromBins = npzdata['maskedChromBins']
    maskedChromBinSums = npzdata['maskedChromBinSums']

    indexes, distances = wisetools.getReference(correctedData, maskedChromBins, maskedChromBinSums,
                                                selectRefAmount=args.refsize, part=args.part[0],
                                                splitParts=args.part[1], device=device)

    np.savez_compressed(args.partfile + '_' + str(args.part[0]) + '.npz',
                        arguments=vars(args),
                        runtime=getRuntime(),
                        indexes=indexes,
                        distances=distances)


def toolNewrefPost(args):
    """reference wisecondor.py:135-170."""
    npzdata = _load(args.prepfile)
    maskedChromBins = npzdata['maskedChromBins']
    chromosomeBins = npzdata['chromosomeBins']
    mask = npzdata['mask']
    pca_components = npzdata['pca_components']
    pca_mean = npzdata['pca_mean']
    binsize = npzdata['binsize'].item()

    bigIndexes = []
    bigDistances = []
    for part in range(1, args.parts + 1):
        infile = args.partfile + '_' + str(part) + '.npz'
        print('Loading:', infile)
        npzdata = _load(infile)
        bigIndexes.append(npzdata['indexes'])
        bigDistances.append(npzdata['distances'])
        print(part, npzdata['indexes'].shape)

    np.savez_compressed(args.outfile,
                        arguments=vars(args),
                        runtime=getRuntime(),
                        binsize=binsize,
                        indexes=np.concatenate(bigIndexes),
                        distances=np.concatenate(bigDistances),
                        chromosome_sizes=chromosomeBins,
                        mask=mask,
                        masked_sizes=maskedChromBins,
                        pca_components=pca_components,
                        pca_mean=pca_mean)


# ---- test -------------------------------------------------------------------------------------------------------------
def _loadReference(path):
    referenceFile = _load(path)
    ref = {key: referenceFile[key] for key in ('indexes', 'distances', 'chromosome_sizes', 'mask', 'masked_sizes',
                                               'pca_mean', 'pca_components')}
    ref['binsize'] = referenceFile['binsize'].item()
    return ref


def _testSamples(samples, sampleBinSizes, ref, args):
    """toolTest's computation (reference wisecondor.py:190-268) for a list of sample dicts; returns one dict of
    result-npz entries per sample."""
    from scipy.special import ndtri          # norm.ppf(q) == ndtri(q) (same Cephes routine), a second less import time
    scaled = [wisetools.scaleSample(s, b, ref['binsize']) for s, b in zip(samples, sampleBinSizes)]
    num_tests = sum(ref['masked_sizes'])
    z_threshold = float(ndtri(1 - 1. / (num_tests * 0.5 * args.multitest)))     # reference wisecondor.py:204
    if args.minzscore is not None:
        z_threshold = args.minzscore
    print('Per bin z-score threshold for first testing cycles:', z_threshold)
    return wisetools.testSamples(scaled, ref, z_threshold, chromosomes=list(args.chromosomes),
                                 mineffectsize=args.mineffectsize, minrefbins=args.minrefbins, repeats=args.repeats)


def _saveResult(outfile, args, binsize, res):
    # np.load reads compressed and stored npz alike; -uncompressed (testbatch) skips zlib, the slowest host step
    save = np.savez if getattr(args, 'uncompressed', False) else np.savez_compressed
    save(outfile,
         arguments=vars(args),
         runtime=getRuntime(),
         binsize=binsize,
         results_r=_ragged(res['results_r']),
         results_z=_ragged(res['results_z']),
         results_cwz=res['results_cwz'],
         results_calls=res['results_calls'],
         threshold_z=res['threshold_z'],
         asdef=res['asdef'],
         aasdef=res['aasdef'])


def toolTest(args):
    """reference wisecondor.py:174-281."""
    ref = _loadReference(args.reference)
    sampleFile = _load(args.infile)
    res, = _testSamples([sampleFile['sample'].item()], [sampleFile['arguments'].item()['binsize']], ref, args)
    print('ASDES:', res['asdef'], '\nAASDEF:', res['aasdef'])
    _saveResult(args.outfile, args, ref['binsize'], res)
    sys.exit(0)


def toolTestBatch(args):
    """Many samples against one reference: device batches of `-batch` samples, one result npz per sample (named after
    the sample file).  npz inflate (loading) and deflate (writing) run in a thread pool and overlap the GPU work of
    the neighbouring batches - at 10 k samples host I/O, not the kernels, sets the pace."""
    import concurrent.futures
    os.makedirs(args.outdir, exist_ok=True)
    gpus = max(1, int(getattr(args, 'gpus', 1) or 1))
    if gpus > 1:
        # samples are independent: shard them over the GPUs, no communication (one process per GPU)
        from wisecondor_b200 import partition
        flags = ['-batch', str(args.batch), '-iothreads', str(args.iothreads), '-chromosomes', ','.join(str(c) for c in args.chromosomes),
                 '-mineffectsize', str(args.mineffectsize), '-multitest', str(args.multitest), '-minrefbins', str(args.minrefbins),
                 '-repeats', str(args.repeats)]
        if args.minzscore is not None:
            flags += ['-minzscore', str(args.minzscore)]
        if args.uncompressed:
            flags.append('-uncompressed')
        procs = []
        for rank in range(gpus):
            a, b = partition.sample_shard(rank, gpus, len(args.infiles))
            if b > a:
                env = dict(os.environ, CUDA_VISIBLE_DEVICES=str(rank))
                procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), 'testbatch'] + list(args.infiles[a:b]) +
                                              [args.outdir, args.reference] + flags, env=env))
        codes = [p.wait() for p in procs]
        if any(codes):
            print('ERROR: worker exit codes', codes)
            sys.exit(1)
        return
    ref = _loadReference(args.reference)

    def load(infile):
        sampleFile = _load(infile)
        return sampleFile['sample'].item(), sampleFile['arguments'].item()['binsize']

    t0 = time.time()
    nbatch = max(1, int(args.batch))
    with concurrent.futures.ThreadPoolExecutor(max_workers=max(2, int(args.iothreads))) as pool:
        loads = [pool.submit(load, f) for f in args.infiles]
        saves = []
        for first in range(0, len(args.infiles), nbatch):
            files = args.infiles[first:first + nbatch]
            loaded = [f.result() for f in loads[first:first + nbatch]]
            results = _testSamples([l[0] for l in loaded], [l[1] for l in loaded], ref, args)
            for infile, res in zip(files, results):
                saves.append(pool.submit(_saveResult, os.path.join(args.outdir, os.path.basename(infile)), args,
                                         ref['binsize'], res))
            for i in range(first, first + len(files)):
                loads[i] = None                      # release the sample dicts
        for f in saves:
            f.result()                               # surface write errors
    print('Time spent on testing', len(args.infiles), 'samples:', round(time.time() - t0, 3), 'seconds')


# ---- host-only tools of the reference that are not part of this build -------------------------------------------------
def _hostOnly(name, why):
    def tool(args):
        print('ERROR: `%s` is a host-only tool of the reference WISECONDOR and is not replaced by this build: %s' % (name, why))
        print('Run it from the reference installation; the npz files are interchangeable.')
        sys.exit(2)
    tool.__name__ = 'tool' + name.capitalize()
    return tool


toolConvert = _hostOnly('convert', 'BAM read-start binning stays on the host (pysam)')
toolPlot = _hostOnly('plot', 'it only reads the result npz (matplotlib)')


def toolReport(args):
    """Text report of one tested sample (reference wisecondor.py:304-342): the arguments of `convert` and `test`, the read
    counts `convert` kept in the sample npz, the z-score threshold and the two sigma averages, and one line per call
    whose effect size exceeds -mineffect percent.  Host only (formatting of two npz files, nothing for the device), the
    same text as the reference prints so that scripts parsing it keep working."""
    sample = _load(args.testfile)
    result = _load(args.resultfile)
    binsize = result['binsize'].item()
    out = []

    def section(title):
        out.append('\n# %s #' % title)

    for title, stored in (('Arguments used in convert:', sample['arguments'].item()),
                          ('Arguments used in test:', result['arguments'].item())):
        section(title)
        out.extend('%s = %s' % (key, stored[key]) for key in stored)

    q = sample['quality'].item()
    section('BAM information:')
    for label, key in (('Reads mapped:  ', 'mapped'), ('Reads unmapped:', 'unmapped'), ('Reads nocoord: ', 'no_coordinate'),
                       ('Reads rmdup:   ', 'filter_rmdup'), ('Reads lowqual: ', 'filter_mapq')):
        out.append('%s\t %s' % (label, q[key]))
    # what went into the tower filter: the reads counted before it, without the coordinate-less ones, with the duplicates
    # and low-quality reads counted back in (the reference's own bookkeeping, wisecondor.py:328-331)
    retro_in = q['pre_retro'] - q['no_coordinate'] + q['filter_rmdup'] + q['filter_mapq']
    section('RETRO filtering:')
    out.append('Reads in:     \t %s' % retro_in)
    out.append('Reads removed:\t %s' % (retro_in - q['post_retro']))
    out.append('Reads out:    \t %s' % q['post_retro'])

    section('Z-Score checks:')
    out.append('Z-Score used:\t %.2f' % result['threshold_z'].item())
    out.append('AvgStdDev:   \t %.2f%%' % (float(result['asdef']) * 100))
    out.append('AvgAllStdDev:\t %.2f%%' % (float(result['aasdef']) * 100))

    section('Test results:')
    out.append('z-score\teffect\tmbsize\tlocation')
    for chrom, first, last, z, effect in result['results_calls']:
        if args.mineffect < abs(effect * 100):
            out.append('%.2f\t%.2f\t%.2f\t%.0f:%.0f-%.0f' % (z, effect * 100, (last - first + 1) * binsize / 1e6, chrom,
                                                            first * binsize, (last + 1) * binsize))
    print('\n'.join(out))


def _intList(text):
    return [int(v) for v in text.split(',')]


def buildParser():
    parser = argparse.ArgumentParser(description="WISECONDOR (WIthin-SamplE COpy Number aberration DetectOR) - B200 build")
    sub = parser.add_subparsers()

    def refsize(text):
        """-refsize: the reference accepts any positive count (wisecondor.py:379); the device search takes up to 4096
        (the wide-refsize search above 384), so larger values are refused HERE, before any work is done."""
        value = int(text)
        if not 1 <= value <= 4096:
            raise argparse.ArgumentTypeError("refsize must be between 1 and 4096 on the B200 search (got %d)" % value)
        return value

    p = sub.add_parser('convert', description='Convert and filter a bam file to an npz')
    p.add_argument('infile', type=str)
    p.add_argument('outfile', type=str)
    p.add_argument('-binsize', type=float, default=1e6)
    p.add_argument('-retdist', type=int, default=4)
    p.add_argument('-retthres', type=int, default=4)
    p.set_defaults(func=toolConvert)

    p = sub.add_parser('newref', description='Create a new reference using healthy reference samples')
    p.add_argument('infiles', type=str, nargs='*', help='Reference sample npz files')
    p.add_argument('outfile', type=str, help='Reference output npz')
    p.add_argument('-refsize', type=refsize, default=100, help='Amount of reference locations per target (1..4096)')
    p.add_argument('-binsize', type=int, default=None, help='Scale samples to this binsize (multiples only)')
    p.add_argument('-cpus', type=int, default=1, help='Kept for compatibility: raises the number of parts')
    p.add_argument('-parts', type=int, default=1, help='Split reference finding in this many row parts')
    p.add_argument('-gpus', type=int, default=1, help='Shard the target bins over this many B200s of the node (one process each, NCCL)')
    p.add_argument('-partfiles', action='store_true', help='With -gpus N: exchange the parts through part files like the reference (resumable per part) instead of NCCL')
    p.set_defaults(func=toolNewref)

    p = sub.add_parser('newrefrank', description='(internal) one rank of newref -gpus N; started once per GPU with RANK / WORLD_SIZE set')
    p.add_argument('prepfile', type=str)
    p.add_argument('outfile', type=str)
    p.add_argument('-refsize', type=refsize, default=100)
    p.set_defaults(func=toolNewrefRank)

    p = sub.add_parser('newrefprep', description='Prepare creation of new reference split over several processes')
    p.add_argument('infiles', type=str, nargs='*')
    p.add_argument('prepfile', type=str)
    p.add_argument('-binsize', type=int, default=None)
    p.set_defaults(func=toolNewrefPrep)

    p = sub.add_parser('newrefpart', description='Creation of new reference split over several processes')
    p.add_argument('prepfile', type=str)
    p.add_argument('partfile', type=str)
    p.add_argument('part', type=int, default=[0, 1], nargs=2)
    p.add_argument('-refsize', type=refsize, default=100)
    p.set_defaults(func=toolNewrefPart)

    p = sub.add_parser('newrefpost', description='Combine creation of new reference split over several processes')
    p.add_argument('prepfile', type=str)
    p.add_argument('partfile', type=str)
    p.add_argument('parts', type=int, default=1)
    p.add_argument('outfile', type=str)
    p.set_defaults(func=toolNewrefPost)

    def testFlags(q):
        q.add_argument('-minzscore', type=float, default=None, help='Minimum absolute z-score')
        q.add_argument('-chromosomes', type=_intList, default=list(range(1, 23)),
                       help='Integer of every chromosome to test, comma delimited')
        q.add_argument('-mineffectsize', type=float, default=0, help='Minimum absolute relative change in read depth')
        q.add_argument('-multitest', type=float, default=1000, help='Compensate the z threshold for multiple testing')
        q.add_argument('-minrefbins', type=int, default=25, help='Minimum amount of sensible ref bins per target bin')
        q.add_argument('-repeats', type=int, default=5, help='Repeats when calling')

    p = sub.add_parser('test', description='Test sample for Copy Number Aberrations')
    p.add_argument('infile', type=str)
    p.add_argument('outfile', type=str)
    p.add_argument('reference', type=str)
    testFlags(p)
    p.set_defaults(func=toolTest)

    p = sub.add_parser('testbatch', description='Test many samples against one reference in one device batch')
    p.add_argument('infiles', type=str, nargs='+')
    p.add_argument('outdir', type=str)
    p.add_argument('reference', type=str)
    testFlags(p)
    p.add_argument('-batch', type=int, default=256, help='Samples per device batch')
    p.add_argument('-iothreads', type=int, default=8, help='Threads loading / writing npz files')
    p.add_argument('-uncompressed', action='store_true', help='Write result npz files without zlib compression')
    p.add_argument('-gpus', type=int, default=1, help='Shard the samples over this many B200s of the node (one process each, no communication)')
    p.set_defaults(func=toolTestBatch)

    p = sub.add_parser('plot', description='Plot results produced by sample testing')
    p.add_argument('infile', type=str)
    p.add_argument('outfile', type=str)
    p.add_argument('-cytofile', type=str, default=None)
    p.add_argument('-chromosomes', type=_intList, default=list(range(1, 23)))
    p.add_argument('-columns', type=int, default=2)
    p.add_argument('-filetype', type=str, default='pdf')
    p.add_argument('-size', type=float, nargs=2, default=[11.7, 8.3])
    p.add_argument('-mineffect', type=float, default=1.5)
    p.set_defaults(func=toolPlot)

    p = sub.add_parser('report', description='Report results produced by sample testing')
    p.add_argument('testfile', type=str)
    p.add_argument('resultfile', type=str)
    p.add_argument('-mineffect', type=float, default=1.5)
    p.set_defaults(func=toolReport)
    return parser


def main(argv=None):
    args = buildParser().parse_args(sys.argv[1:] if argv is None else argv)
    if not hasattr(args, 'func'):
        buildParser().print_help()
        sys.exit(2)
    printArgs(args)
    before = _mem.BACKEND
    if 'WISECONDOR_BACKEND' not in os.environ:
        # Device buffers: `testbatch` pipelines chunks over torch streams and pinned memory; everything else handles one
        # reference or one sample and takes the library's own cudaMalloc buffers - importing PyTorch alone would cost
        # more than their whole run.
        _mem.BACKEND = 'torch' if args.func in (toolTestBatch, toolNewrefRank) else 'native'
    try:
        args.func(args)
    finally:
        _mem.BACKEND = before            # main() may be called in-process (tests, notebooks): leave no global behind


if __name__ == '__main__':
    main()
