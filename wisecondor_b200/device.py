"""Device-resident entry points: device arrays own the HBM buffers, the C ABI does the work.

The arrays are torch CUDA tensors (library use: streams, pinned memory, torch.distributed) or _mem.DevArray blocks
(the command line without PyTorch); every function returns the kind it was given.  Either way this is plumbing: every
kernel lives in libwisecondor_b200.so.
"""
import ctypes

import numpy as np

from . import _cabi, _mem
from ._mem import ptr as _ptr, stream_ptr as _stream_ptr, require as _require_cuda

F64, I32, U8 = np.float64, np.int32, np.uint8


def newref_topk(corrected, chrom_bins, row_begin, row_end, refsize, out_idx=None, out_dist=None):
    """Reference-bin search for target rows [row_begin, row_end) (wisetools.py:364-398, 298-325).

    corrected: CUDA float64 [N][S] (bin-major).  Returns (indexes int32 [rows][refsize], distances float64
    [rows][refsize]) on the same device; indexes are positions in the other-chromosome concatenation.
    """
    _require_cuda(corrected, F64, "corrected")
    n, s = corrected.shape
    cb = np.ascontiguousarray(chrom_bins, dtype=np.int32)
    rows = int(row_end) - int(row_begin)
    if out_idx is None:
        out_idx = _mem.empty((max(rows, 0), refsize), I32, like=corrected)
    if out_dist is None:
        out_dist = _mem.empty((max(rows, 0), refsize), F64, like=corrected)
    ctx = _cabi.context(_mem.device_index(corrected))
    rc = _cabi.lib().wc_newref_topk(ctx.handle, _ptr(corrected), n, s, cb.ctypes.data_as(ctypes.c_void_p), len(cb),
                                    int(row_begin), int(row_end), int(refsize), _ptr(out_idx), _ptr(out_dist),
                                    _stream_ptr(corrected))
    _cabi.check(rc)
    return out_idx, out_dist


def newref_topk_host(corrected, chrom_bins, row_begin, row_end, refsize, device=0, out_idx=None, out_dist=None):
    """Same search with HOST numpy buffers: copies in and out inside the C call (wc_newref_topk_host).  out_idx /
    out_dist may be preallocated (e.g. views of pinned memory: faster device-to-host copies)."""
    X = np.ascontiguousarray(corrected, dtype=np.float64)
    n, s = X.shape
    cb = np.ascontiguousarray(chrom_bins, dtype=np.int32)
    rows = int(row_end) - int(row_begin)
    idx = np.empty((max(rows, 0), refsize), dtype=np.int32) if out_idx is None else out_idx
    dist = np.empty((max(rows, 0), refsize), dtype=np.float64) if out_dist is None else out_dist
    if idx.shape != (max(rows, 0), refsize) or idx.dtype != np.int32 or not idx.flags.c_contiguous or \
            dist.shape != idx.shape or dist.dtype != np.float64 or not dist.flags.c_contiguous:
        raise _cabi.WisecondorError("out_idx / out_dist must be C-contiguous int32 / float64 arrays of shape rows x refsize")
    ctx = _cabi.context(device)
    rc = _cabi.lib().wc_newref_topk_host(ctx.handle, X.ctypes.data_as(ctypes.c_void_p), n, s,
                                         cb.ctypes.data_as(ctypes.c_void_p), len(cb), int(row_begin), int(row_end),
                                         int(refsize), idx.ctypes.data_as(ctypes.c_void_p),
                                         dist.ctypes.data_as(ctypes.c_void_p))
    _cabi.check(rc)
    return idx, dist


# ---- sharded symmetric search: the three steps of one rank (wisecondor_b200.shard.SymmetricShardedSearch drives them) ----
I64 = np.int64


def shard_dims(n, refsize, world, rank, device=0, ctx=None):
    """Sizes of the exchange buffers of a sharded symmetric search (wc_newref_shard_dims)."""
    ctx = ctx or _cabi.context(device)
    out = (ctypes.c_longlong * 6)()
    _cabi.check(_cabi.lib().wc_newref_shard_dims(ctx.handle, int(n), int(refsize), int(world), int(rank), out))
    return {"rows_per": int(out[0]), "in_cap": int(out[1]), "thr_len": int(out[2]), "row0": int(out[3]),
            "row1": int(out[4]), "blocks": int(out[5])}


def shard_begin(corrected, chrom_bins, refsize, rank, world, thr, ctx=None):
    """K4 + threshold pass over this rank's row blocks; thr: device int64 [thr_len] (u64 keys), written."""
    _require_cuda(corrected, F64, "corrected")
    _require_cuda(thr, I64, "thr")
    n, s = corrected.shape
    cb = np.ascontiguousarray(chrom_bins, dtype=np.int32)
    ctx = ctx or _cabi.context(_mem.device_index(corrected))
    _cabi.check(_cabi.lib().wc_newref_shard_begin(ctx.handle, _ptr(corrected), n, s, cb.ctypes.data_as(ctypes.c_void_p), len(cb),
                                                  int(refsize), int(rank), int(world), _ptr(thr), _stream_ptr(corrected)))


def shard_sweep(thr, in_key, in_j, in_cnt, ctx=None):
    """Symmetric pass; thr after the all-reduce(MIN); in_key int64 / in_j int32 [world*rows_per][in_cap], in_cnt int32."""
    _require_cuda(thr, I64, "thr")
    _require_cuda(in_key, I64, "in_key")
    _require_cuda(in_j, I32, "in_j")
    _require_cuda(in_cnt, I32, "in_cnt")
    ctx = ctx or _cabi.context(_mem.device_index(thr))
    _cabi.check(_cabi.lib().wc_newref_shard_sweep(ctx.handle, _ptr(thr), _ptr(in_key), _ptr(in_j), _ptr(in_cnt), _stream_ptr(thr)))


def shard_finish(recv_key, recv_j, recv_cnt, out_idx, out_dist, ctx=None):
    """Exact re-score and ranking of this rank's bins from its own segments and the received column-side candidates."""
    _require_cuda(recv_key, I64, "recv_key")
    _require_cuda(recv_j, I32, "recv_j")
    _require_cuda(recv_cnt, I32, "recv_cnt")
    _require_cuda(out_idx, I32, "out_idx")
    _require_cuda(out_dist, F64, "out_dist")
    ctx = ctx or _cabi.context(_mem.device_index(recv_key))
    _cabi.check(_cabi.lib().wc_newref_shard_finish(ctx.handle, _ptr(recv_key), _ptr(recv_j), _ptr(recv_cnt), _ptr(out_idx),
                                                   _ptr(out_dist), _stream_ptr(recv_key)))
    return out_idx, out_dist


def last_search_stats(device=0):
    """Device timings (ms) and counters of the most recent search on `device`."""
    ctx = _cabi.context(device)
    return {
        "center_norms_ms": ctx.phase_ms(0), "dist_topk_ms": ctx.phase_ms(1), "finalize_ms": ctx.phase_ms(2),
        "dist_topk_first_pass_ms": ctx.phase_ms(8),
        "finalize_rescore_ms": ctx.phase_ms(10),       # K6 split form: the streaming exact re-score alone (0: fused kernel)
        "exhaustive_ms": ctx.phase_ms(3), "launches": ctx.counter(0), "exhaustive_rows": ctx.counter(1),
        "tiles": ctx.counter(3), "tiles_plain": ctx.counter(2), "ctas": ctx.counter(4),
        "filter": max(0, ctx.counter(7)) & 3,          # 0: fp64 DMMA, 1: fp16 mma.sync, 2: fp16 tcgen05 / TMEM
        "pivots": max(0, ctx.counter(7)) >> 4,         # pivots of the K5t pivot pass (0: none)
        "k6_live_entries": ctx.counter(8),             # K6 split form: entries within the rows' final thresholds, all rows
        "k6_shortlisted": ctx.counter(9),              # ... and candidates re-scored exactly (0: fused kernel)
        "k6_live_max": ctx.counter(11),                # most live entries of one row among the warp-selected rows
        "k6_rows_cta_select": ctx.counter(10),         # rows the warp-per-row select passed on to the CTA-per-row one
    }


# ------------------------------------------------------------------------------------------------------------
# test: batched sample preparation, z-scores, segmentation
# ------------------------------------------------------------------------------------------------------------
CALL_DTYPE = np.dtype([("sample", np.int32), ("chrom", np.int32), ("x", np.int32), ("y", np.int32), ("z", np.float64)])


def _ints(values):
    arr = np.ascontiguousarray(values, dtype=np.int32)
    return arr, arr.ctypes.data_as(ctypes.c_void_p)


def pad32(b):
    return (int(b) + 31) // 32 * 32


class ReferenceTable(object):
    """Device-resident form of a reference npz for the test path: per bin the global ids of its usable reference
    bins (`index[distances < cutoff]` mapped out of other-chromosome coordinates, wisetools.py:420-424).  Any refsize
    with N x wc_table_stride(refsize) < 2^31 is accepted; the table and the reverse table take 2 x N x stride x 4 B
    of device memory (1.9 GB at 50 kb with refsize 4096)."""

    def __init__(self, indexes, distances, masked_sizes, cutoff, device=0):
        self.masked_sizes = [int(v) for v in masked_sizes]
        self.n, self.k = int(indexes.shape[0]), int(indexes.shape[1])
        stride = _cabi.lib().wc_table_stride(self.k)
        if self.n * stride >= 2 ** 31:
            raise _cabi.WisecondorError("reference table of %d bins x refsize %d (row stride %d) needs N x stride < 2^31"
                                        % (self.n, self.k, stride))
        self.cutoff = float(cutoff)
        idx = _mem.to_device(np.ascontiguousarray(indexes, dtype=np.int32), device)
        dst = _mem.to_device(np.ascontiguousarray(distances, dtype=np.float64), device)
        self.device = idx.device
        self.table = _mem.empty((self.n, stride), I32, like=idx)
        self.count = _mem.empty((self.n,), I32, like=idx)
        # reverse table (CSR): which bins use bin j as a reference bin
        self.rev_off = _mem.empty((self.n + 1,), I32, like=idx)
        self.rev_idx = _mem.empty((self.n, self.table.shape[1]), I32, like=idx)
        cb, cbp = _ints(self.masked_sizes)
        ctx = _cabi.context(_mem.device_index(idx))
        rc = _cabi.lib().wc_test_table(ctx.handle, _ptr(idx), _ptr(dst), self.n, self.k, cbp, len(cb), self.cutoff,
                                       _ptr(self.table), _ptr(self.count), _ptr(self.rev_off), _ptr(self.rev_idx),
                                       _stream_ptr(idx))
        _cabi.check(rc)
        _mem.synchronize(idx)


def test_prep(counts, masked_raw, pca_mean, pca_components, nsamples=None):
    """toNumpyRefFormat's normalise+mask and applyPCA (wisetools.py:275-276, 104-113) for a batch.

    counts: CUDA int32 [B][Nraw] (chromosomes already padded/truncated to the reference sizes); masked_raw: CUDA
    int32 [N]; pca_mean CUDA f64 [N]; pca_components CUDA f64 [ncomp][N].  Returns T: CUDA f64 [N][pad32(B)]."""
    _require_cuda(counts, I32, "counts")
    _require_cuda(masked_raw, I32, "masked_raw")
    b, nraw = counts.shape
    n = masked_raw.shape[0]
    dev = counts          # outputs follow its kind, device and stream
    if pca_components is None:        # normalise + mask only (toNumpyRefFormat)
        ncomp = 0
        pca_mean = pca_components = _mem.empty((0,), F64, like=dev)
    else:
        _require_cuda(pca_mean, F64, "pca_mean")
        _require_cuda(pca_components, F64, "pca_components")
        ncomp = pca_components.shape[0]
    ldb = pad32(b)
    out = _mem.empty((n, ldb), F64, like=dev)
    ctx = _cabi.context(_mem.device_index(dev))
    rc = _cabi.lib().wc_test_prep(ctx.handle, _ptr(counts), b, nraw, _ptr(masked_raw), n, _ptr(pca_mean),
                                  _ptr(pca_components), ncomp, _ptr(out), ldb, _stream_ptr(dev))
    _cabi.check(rc)
    return out


def apply_pca(x, pca_mean, pca_components):
    """applyPCA (wisetools.py:104-113) for a batch of normalised masked vectors x: CUDA f64 [B][N].
    Returns T: CUDA f64 [N][pad32(B)] (sample-minor)."""
    _require_cuda(x, F64, "x")
    _require_cuda(pca_mean, F64, "pca_mean")
    _require_cuda(pca_components, F64, "pca_components")
    b, n = x.shape
    dev = x          # outputs follow its kind, device and stream
    ldb = pad32(b)
    out = _mem.empty((n, ldb), F64, like=dev)
    ctx = _cabi.context(_mem.device_index(dev))
    rc = _cabi.lib().wc_apply_pca(ctx.handle, _ptr(x), b, n, _ptr(pca_mean), _ptr(pca_components),
                                  pca_components.shape[0], _ptr(out), ldb, _stream_ptr(dev))
    _cabi.check(rc)
    return out


def zscore_batch(test, nsamples, table, z_threshold, repeats, copy_init=None):
    """repeatTest (wisetools.py:438-448) for a batch.  test: CUDA f64 [N][ldb] sample-minor; table: ReferenceTable;
    copy_init: optional CUDA f64 [N][ldb], trySample's pre-marked `testCopy`.
    Returns (z [B][N], r [B][N], refsizes int32 [B][N], asdef [B]) on the device."""
    _require_cuda(test, F64, "test")
    if copy_init is not None:
        _require_cuda(copy_init, F64, "copy_init")
        if copy_init.shape != test.shape:
            raise _cabi.WisecondorError("copy_init must have the shape of test")
    n, ldb = test.shape
    b = int(nsamples)
    dev = test          # outputs follow its kind, device and stream
    z = _mem.empty((b, n), F64, like=dev)
    r = _mem.empty((b, n), F64, like=dev)
    sizes = _mem.empty((b, n), I32, like=dev)
    asdef = _mem.empty((b,), F64, like=dev)
    ctx = _cabi.context(_mem.device_index(dev))
    rc = _cabi.lib().wc_zscore_batch(ctx.handle, _ptr(test), _ptr(copy_init) if copy_init is not None else None, n, b, ldb,
                                     _ptr(table.table), _ptr(table.count), _ptr(table.rev_off), _ptr(table.rev_idx), table.k,
                                     float(z_threshold), int(repeats), _ptr(z), _ptr(r), _ptr(sizes), _ptr(asdef),
                                     _stream_ptr(dev))
    _cabi.check(rc)
    return z, r, sizes, asdef


def segment_batch(z, refsizes, masked_sizes, chromosomes, minrefbins, z_threshold, min_search=3, max_calls=256, r=None,
                  mineffectsize=0.0):
    """The chromosome loop of toolTest (wisecondor.py:233-238) for a batch.  z: CUDA f64 [B][N]; refsizes: CUDA
    int32 [B][N]; chromosomes: 0-based indices; r (CUDA f64 [B][N], resultsR) and mineffectsize select fillTriMin's
    effect-size filter (wisetools.py:475-487).  Returns (cwz [B][nsel] CUDA, cleaned_bins int32 [B][nsel] CUDA,
    calls: numpy structured array (sample, chrom, x, y, z) sorted by (sample, chrom, x))."""
    _require_cuda(z, F64, "z")
    _require_cuda(refsizes, I32, "refsizes")
    if mineffectsize != 0:
        _require_cuda(r, F64, "r")
        if r.shape != z.shape:
            raise _cabi.WisecondorError("r must have the shape of z")
    b, n = z.shape
    dev = z          # outputs follow its kind, device and stream
    cb, cbp = _ints(masked_sizes)
    sel, selp = _ints(chromosomes)
    cwz = _mem.empty((b, len(sel)), F64, like=dev)
    cleaned = _mem.empty((b, len(sel)), I32, like=dev)
    ctx = _cabi.context(_mem.device_index(dev))
    while True:
        calls = _mem.empty((b, max_calls * CALL_DTYPE.itemsize), U8, like=dev)
        ncalls = _mem.empty((b,), I32, like=dev)
        rc = _cabi.lib().wc_segment_batch(ctx.handle, _ptr(z), _ptr(r) if r is not None else None, _ptr(refsizes), n, b,
                                          cbp, len(cb), selp, len(sel), int(minrefbins), float(z_threshold),
                                          float(mineffectsize), int(min_search), _ptr(cwz), _ptr(cleaned),
                                          _ptr(calls), _ptr(ncalls), int(max_calls), _stream_ptr(dev))
        if rc != 0 and b"max_calls" in _cabi.lib().wc_last_error() and max_calls < (1 << 16):
            max_calls *= 8
            continue
        _cabi.check(rc)
        break
    nc = _mem.to_host(ncalls)
    raw = _mem.to_host(calls).view(CALL_DTYPE).reshape(b, max_calls)
    rows = [raw[i, :nc[i]] for i in range(b)]
    flat = np.concatenate(rows) if rows else np.zeros(0, dtype=CALL_DTYPE)
    flat = flat[np.lexsort((flat["x"], flat["chrom"], flat["sample"]))]
    return cwz, cleaned, flat


def last_test_stats(device=0):
    """Device timings (ms) of the most recent prep / z-score / segmentation calls on `device`."""
    ctx = _cabi.context(device)
    pairs = []
    while len(pairs) < 64:
        n = ctx.counter(16 + len(pairs))
        if n < 0:
            break
        pairs.append(int(n))
    return {"prep_ms": ctx.phase_ms(6), "zscore_ms": ctx.phase_ms(4), "segment_ms": ctx.phase_ms(5),
            "zscore_launches": ctx.counter(5), "segment_launches": ctx.counter(6), "zscore_pairs_per_pass": pairs}


# ------------------------------------------------------------------------------------------------------------
# newref preparation: normalise, mask, PCA residual
# ------------------------------------------------------------------------------------------------------------
def newref_normalize(counts):
    """toNumpyArray's arithmetic (wisetools.py:255-261).  counts: CUDA int32 [S][Nraw].
    Returns (maskedData CUDA f64 [N][S] bin-major, mask numpy bool [Nraw])."""
    _require_cuda(counts, I32, "counts")
    s, nraw = counts.shape
    dev = counts          # outputs follow its kind, device and stream
    ctx = _cabi.context(_mem.device_index(dev))
    mask_d = _mem.empty((nraw,), U8, like=dev)
    _cabi.check(_cabi.lib().wc_newref_mask(ctx.handle, _ptr(counts), s, nraw, _ptr(mask_d), _stream_ptr(dev)))
    mask = _mem.to_host(mask_d).astype(bool)
    masked_raw = _mem.to_device(np.flatnonzero(mask).astype(np.int32), like=dev)
    n = int(masked_raw.shape[0])
    masked = _mem.empty((n, s), F64, like=dev)
    if n > 0:
        _cabi.check(_cabi.lib().wc_newref_normalize(ctx.handle, _ptr(counts), s, nraw, _ptr(masked_raw), n, _ptr(masked),
                                                    _stream_ptr(dev)))
    return masked, mask


def top_eigenpairs(gram, ncomp):
    """Largest `ncomp` eigenpairs of the symmetric S x S Gram matrix (host LAPACK; the only N-independent step
    of the PCA).  Returns (eigenvectors S x ncomp, largest first; singular values = sqrt(eigenvalues))."""
    s = gram.shape[0]
    try:
        from scipy.linalg import eigh
        w, v = eigh(gram, subset_by_index=[max(0, s - ncomp), s - 1])
    except ImportError:                                   # pragma: no cover
        w, v = np.linalg.eigh(gram)
        w, v = w[-ncomp:], v[:, -ncomp:]
    order = np.argsort(w)[::-1]
    w, v = w[order], v[:, order]
    return np.ascontiguousarray(v), np.sqrt(np.maximum(w, 0.0))


def pca_fit_apply(masked, ncomp=3):
    """trainPCA (wisetools.py:89-101) with the exact top-`ncomp` principal subspace.  masked: CUDA f64 [N][S].
    Returns (corrected CUDA f64 [N][S], components numpy [ncomp][N] with scikit-learn's sign convention,
    mean numpy [N])."""
    _require_cuda(masked, F64, "masked")
    n, s = masked.shape
    dev = masked          # outputs follow its kind, device and stream
    ctx = _cabi.context(_mem.device_index(dev))
    mean = _mem.empty((n,), F64, like=dev)
    gram = _mem.empty((s, s), F64, like=dev)
    _cabi.check(_cabi.lib().wc_pca_gram(ctx.handle, _ptr(masked), n, s, _ptr(mean), _ptr(gram), _stream_ptr(dev)))
    vec, sigma = top_eigenpairs(_mem.to_host(gram), ncomp)
    if not (sigma > 0).all():
        raise _cabi.WisecondorError("PCA: fewer than %d non-zero singular values (degenerate sample matrix)" % ncomp)
    vec_d = _mem.to_device(vec, like=dev)
    comps = _mem.empty((ncomp, n), F64, like=dev)
    corrected = _mem.empty((n, s), F64, like=dev)
    sig = np.ascontiguousarray(sigma, dtype=np.float64)
    _cabi.check(_cabi.lib().wc_pca_apply(ctx.handle, _ptr(masked), n, s, _ptr(mean), _ptr(vec_d),
                                         sig.ctypes.data_as(ctypes.c_void_p), ncomp, _ptr(comps), _ptr(corrected),
                                         _stream_ptr(dev)))
    comps_h = _mem.to_host(comps)
    # scikit-learn svd_flip(u_based_decision=False): the largest-magnitude entry of every component is positive
    signs = np.sign(comps_h[np.arange(ncomp), np.argmax(np.abs(comps_h), axis=1)])
    signs[signs == 0] = 1.0
    return corrected, comps_h * signs[:, None], _mem.to_host(mean)
