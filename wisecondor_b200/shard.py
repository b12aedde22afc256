"""Partitioning of the hot path over the GPUs of one node (one process per GPU, torch.distributed).

newref: target-bin rows are sharded with the reference's own getPart (wisetools.py:358-361) - rank r of W computes
exactly what `newrefpart r+1 W` would - every rank holds the full corrected matrix, and one all-gather of the
(rows x refsize) int32 + float64 blocks replaces toolNewrefPost's file concatenation (wisecondor.py:146-158).
test: samples are sharded; no communication.  Works with the nccl backend (CUDA tensors) and gloo (CPU tensors; used
by the CPU tests).

SymmetricShardedSearch divides the BLOCK PAIRS of the symmetric search over the ranks instead (every unordered pair of
128-bin blocks is contracted once in the whole job); it has the path's one real exchange step: an all-reduce(MIN) of
the bins' thresholds after the first pass and an all-to-all of the column-side candidates before the final ranking.
"""
import torch
import torch.distributed as dist


from .partition import max_shard_rows, row_shard, sample_shard  # noqa: E402,F401  (torch-free definitions)


class RowGather(object):
    """Buffers of the rows' all-gather: a rank's (rows x k) int32 indexes and float64 distances live side by side in ONE
    byte block (padded to the largest part), so the gather is ONE collective (all_gather_into_tensor); `idx_local` /
    `dist_local` are views of this rank's block - a search that writes into them needs no staging copy."""

    def __init__(self, bincount, k, world, device):
        self.bincount, self.k, self.world = int(bincount), int(k), int(world)
        self.rmax = max_shard_rows(world, bincount)
        self.ib = (self.rmax * self.k * 4 + 15) // 16 * 16               # the distances start 16-byte aligned
        self.db = self.rmax * self.k * 8
        self.block = self.ib + self.db
        self.local = torch.empty(self.block, dtype=torch.uint8, device=device)
        self.all = torch.empty(world * self.block, dtype=torch.uint8, device=device)
        self.idx_local, self.dist_local = self._views(self.local, 0)
        self.lens = [row_shard(r, world, bincount)[1] - row_shard(r, world, bincount)[0] for r in range(world)]

    def _views(self, buf, r):
        o = r * self.block
        idx = buf[o:o + self.rmax * self.k * 4].view(torch.int32).view(self.rmax, self.k)
        dst = buf[o + self.ib:o + self.ib + self.db].view(torch.float64).view(self.rmax, self.k)
        return idx, dst

    def gather(self, group=None, out_idx=None, out_dist=None):
        dist.all_gather_into_tensor(self.all, self.local, group=group)
        if out_idx is None:
            out_idx = torch.empty((self.bincount, self.k), dtype=torch.int32, device=self.local.device)
            out_dist = torch.empty((self.bincount, self.k), dtype=torch.float64, device=self.local.device)
        parts = [self._views(self.all, r) for r in range(self.world)]
        torch.cat([parts[r][0][:self.lens[r]] for r in range(self.world)], out=out_idx)       # drop the padding rows
        torch.cat([parts[r][1][:self.lens[r]] for r in range(self.world)], out=out_dist)
        return out_idx, out_dist


def allgather_rows(idx_local, dist_local, bincount, group=None, out_idx=None, out_dist=None, scratch=None):
    """Concatenate every rank's (rows x k) result block in rank order -> (bincount x k) on every rank.

    Parts differ by at most one row, so blocks are padded to the largest part; indexes and distances travel in one
    collective (RowGather).  `scratch` may carry a RowGather whose idx_local / dist_local the search wrote into."""
    world = dist.get_world_size(group)
    k = idx_local.shape[1]
    rg = scratch if isinstance(scratch, RowGather) else RowGather(bincount, k, world, idx_local.device)
    rows = idx_local.shape[0]
    if rg.idx_local.data_ptr() != idx_local.data_ptr():
        rg.idx_local[:rows].copy_(idx_local)
    if rg.dist_local.data_ptr() != dist_local.data_ptr():
        rg.dist_local[:rows].copy_(dist_local)
    return rg.gather(group=group, out_idx=out_idx, out_dist=out_dist)


class ShardedSearch(object):
    """newref search of one matrix on all ranks of the group, from HOST buffers (the multi-GPU form of
    device.newref_topk_host).  Every rank uploads only its slice of the corrected matrix over PCIe; one NCCL
    all-gather over NVLink assembles the full matrix on every GPU (277 MB at 600 x 50 kb: < 1 ms, against ~9 ms
    for eight simultaneous full uploads); each rank then searches its getPart rows and copies them back to (pinned)
    host memory - the counterpart of the reference's per-part npz files (wisecondor.py:128-132)."""

    def __init__(self, n, s, refsize, rank, world, device, group=None, symmetric=False):
        from . import device as _dev
        self._dev = _dev
        self.n, self.s, self.k, self.rank, self.world, self.group = int(n), int(s), int(refsize), rank, world, group
        self.device = device
        self.rows_per = (self.n + world - 1) // world                 # matrix slices: equal, padded
        self.local = torch.empty((self.rows_per, self.s), dtype=torch.float64, device=device)
        self.full = torch.empty((world * self.rows_per, self.s), dtype=torch.float64, device=device)
        self.r0, self.r1 = row_shard(rank, world, self.n)            # search rows: the reference's getPart
        self.sym = None
        if symmetric and self.k > _dev.NARROW_REFSIZE_MAX:
            raise ValueError("the symmetric sharded search takes refsize up to %d (got %d): use row shards"
                             % (_dev.NARROW_REFSIZE_MAX, self.k))
        if symmetric:        # block pairs instead of rows: this rank's bins are the blocks it owns (SymmetricShardedSearch)
            self.sym = SymmetricShardedSearch(self.n, self.k, rank, world, device, group=group)
            self.r0, self.r1 = self.sym.row0, max(self.sym.row0, self.sym.row1)
        rows = self.r1 - self.r0
        self.idx = torch.empty((rows, self.k), dtype=torch.int32, device=device)
        self.dist = torch.empty((rows, self.k), dtype=torch.float64, device=device)
        self.h_idx = torch.empty((rows, self.k), dtype=torch.int32).pin_memory()
        self.h_dist = torch.empty((rows, self.k), dtype=torch.float64).pin_memory()

    def run(self, x_host, chrom_bins):
        """x_host: pinned CPU tensor [N][S] float64 (every rank holds it, reads only its slice).  Returns this rank's
        rows (indexes, distances) as numpy views of pinned memory."""
        a = self.rank * self.rows_per
        b = min(self.n, a + self.rows_per)
        if b > a:
            self.local[:b - a].copy_(x_host[a:b], non_blocking=True)
        if self.world > 1:
            dist.all_gather_into_tensor(self.full, self.local, group=self.group)
            x = self.full[:self.n]
        else:
            x = self.local[:self.n]
        if self.sym is not None:
            self.idx, self.dist = self.sym.run(x, chrom_bins)
        else:
            self._dev.newref_search(x, chrom_bins, self.r0, self.r1, self.k, out_idx=self.idx, out_dist=self.dist)
        self.h_idx.copy_(self.idx, non_blocking=True)
        self.h_dist.copy_(self.dist, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return self.h_idx.numpy(), self.h_dist.numpy()


class _DeviceEngine(object):
    """The three C-ABI steps of one rank (device.shard_*).  Tests substitute a CPU stand-in to exercise the collectives."""

    def __init__(self, ctx=None):
        from . import device as _dev
        self._dev, self._ctx = _dev, ctx

    def dims(self, n, refsize, world, rank, device):
        index = device.index if getattr(device, "index", None) is not None else 0
        return self._dev.shard_dims(n, refsize, world, rank, device=index, ctx=self._ctx)

    def begin(self, x, chrom_bins, refsize, rank, world, thr):
        self._dev.shard_begin(x, chrom_bins, refsize, rank, world, thr, ctx=self._ctx)

    def sweep(self, thr, in_key, in_j, in_cnt):
        self._dev.shard_sweep(thr, in_key, in_j, in_cnt, ctx=self._ctx)

    def finish(self, recv_key, recv_j, recv_cnt, idx, dist_out):
        self._dev.shard_finish(recv_key, recv_j, recv_cnt, idx, dist_out, ctx=self._ctx)


class SymmetricShardedSearch(object):
    """newref search of one device-resident matrix on all ranks of the group with the symmetric search
    (wc_newref_shard_*, include/wisecondor_b200.h): rank r owns blocks_per = ceil(blocks / world) consecutive 128-bin
    blocks, computes the tiles whose row block it owns and finalises its own bins.  run() returns this rank's rows;
    gather() the whole (N x refsize) result on every rank."""

    def __init__(self, n, refsize, rank, world, device, group=None, engine=None):
        self.n, self.k, self.rank, self.world, self.group, self.device = int(n), int(refsize), rank, world, group, device
        self.engine = engine or _DeviceEngine()
        d = self.engine.dims(self.n, self.k, world, rank, device)
        self.rows_per, self.in_cap, self.row0, self.row1 = d["rows_per"], d["in_cap"], d["row0"], d["row1"]
        total = world * self.rows_per
        self.thr = torch.empty((d["thr_len"],), dtype=torch.int64, device=device)
        self.in_key = torch.empty((total, self.in_cap), dtype=torch.int64, device=device)
        self.in_j = torch.empty((total, self.in_cap), dtype=torch.int32, device=device)
        self.in_cnt = torch.empty((total,), dtype=torch.int32, device=device)
        if world > 1:
            self.recv_key, self.recv_j, self.recv_cnt = (torch.empty_like(t) for t in (self.in_key, self.in_j, self.in_cnt))
        else:
            self.recv_key, self.recv_j, self.recv_cnt = self.in_key, self.in_j, self.in_cnt
        rows = max(0, self.row1 - self.row0)
        self.idx = torch.empty((rows, self.k), dtype=torch.int32, device=device)
        self.dist = torch.empty((rows, self.k), dtype=torch.float64, device=device)
        self._gather = None

    def run(self, x, chrom_bins):
        """x: the whole corrected matrix [N][S] on this rank's device.  Returns (indexes, distances) of the bins
        [row0, row1) this rank owns."""
        self.engine.begin(x, chrom_bins, self.k, self.rank, self.world, self.thr)
        if self.world > 1:
            dist.all_reduce(self.thr, op=dist.ReduceOp.MIN, group=self.group)       # every bin's threshold, everywhere
        self.engine.sweep(self.thr, self.in_key, self.in_j, self.in_cnt)
        if self.world > 1:                                                            # candidates travel to the bins' owners
            dist.all_to_all_single(self.recv_cnt, self.in_cnt, group=self.group)
            dist.all_to_all_single(self.recv_key, self.in_key, group=self.group)
            dist.all_to_all_single(self.recv_j, self.in_j, group=self.group)
        self.engine.finish(self.recv_key, self.recv_j, self.recv_cnt, self.idx, self.dist)
        return self.idx, self.dist

    def gather(self):
        """All ranks' rows in order -> (N x refsize) indexes and distances on every rank."""
        if self.world == 1:
            return self.idx, self.dist
        if self._gather is None:
            self._gather = (torch.zeros((self.rows_per, self.k), dtype=torch.int32, device=self.device),
                            torch.zeros((self.rows_per, self.k), dtype=torch.float64, device=self.device),
                            torch.empty((self.world * self.rows_per, self.k), dtype=torch.int32, device=self.device),
                            torch.empty((self.world * self.rows_per, self.k), dtype=torch.float64, device=self.device))
        pad_i, pad_d, all_i, all_d = self._gather
        pad_i[:self.idx.shape[0]].copy_(self.idx)
        pad_d[:self.dist.shape[0]].copy_(self.dist)
        dist.all_gather_into_tensor(all_i, pad_i, group=self.group)
        dist.all_gather_into_tensor(all_d, pad_d, group=self.group)
        return all_i[:self.n], all_d[:self.n]           # owned ranges are consecutive: rank r holds rows [r*rows_per, ...)
