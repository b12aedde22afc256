#!/usr/bin/env python
"""bench.py - newref reference-bin search throughput (bin-pairs/s) on B200, beside the reference's CPU path.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on
rank 0.  A *step* is one full pass of the hot path - K4 centre+norms, K5 fp64 DMMA distance tiles with the
fused streaming top-k, K6 exact re-score/finalise, and for N > 1 the NCCL all-gather of the row shards - over
a synthetic corrected sample x bin matrix of the named workload, inputs resident in HBM.

  value     whole-job bin-pairs/s = (N^2 - sum N_c^2) / max-over-ranks device time per step
  roofline  the dominant kernel (K5): 2*S*pairs flops per launch / its CUDA-event duration, against the FP64
            tensor-core peak measured on this pool (profiles/fp64_peak_r01.json; MEASURED_PEAKS.json carries
            no FP64 figure)
  e2e       the same metric through the host-buffer C-ABI call (pinned host -> device copy of the matrix and
            device -> host copy of the result inside the timed region)
  cpu_baseline / --impl reference   the reference's own numpy path (oracle/_ref, generated from
            /root/reference by oracle/make_ref.py) on all host cores, on a bounded slice of target rows;
            falls back to the C port of the oracle when oracle/_ref did not travel.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from wisecondor_b200 import synth  # noqa: E402

WORKLOADS = {
    # name: (binsize, samples, refsize, BASELINE.json config it corresponds to)
    "newref_600x250kb": (250000, 600, 100, "configs[1]"),
    "newref_600x50kb": (50000, 600, 100, "configs[2]"),
    "newref_2000x10kb": (10000, 2000, 100, "configs[4]"),
    "newref_20x250kb": (250000, 20, 100, "configs[0]"),
}
DEFAULT_WORKLOAD = "newref_600x50kb"
METRIC = "newref_bin_pairs_per_s"
UNIT = "bin-pairs/s"
# --dump-outputs: the search table and the test path's per-bin vectors, sampled to these sizes in float64 (with the test
# batch's chromosome-wide z-scores, sigma averages and calls the dump stays below 64 MB)
DUMP_TABLE_BYTES = 40 * 10**6
DUMP_TEST_BYTES = 16 * 10**6


def pairs_for_rows(bins, r0, r1):
    n = int(sum(bins))
    per_row = n - np.repeat(np.asarray(bins, dtype=np.int64), bins)
    return int(per_row[r0:r1].sum())


def get_part(partnum, outof, bincount):
    return int(bincount / float(outof) * partnum), int(bincount / float(outof) * (partnum + 1))


def _sample_rows(n, keep):
    """All of range(n), or `keep` of them drawn with a fixed seed: two builds dump the same rows."""
    return np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))


def dump_outputs(path, table_idx, table_dist):
    """The reference-bin table (what a reference npz stores as `indexes` / `distances`) as float64 .npy files."""
    n, k = table_idx.shape
    rows = _sample_rows(n, DUMP_TABLE_BYTES // (16 * k))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "indexes.npy"), table_idx.cpu().numpy()[rows].astype(np.float64))
    np.save(os.path.join(path, "distances.npy"), table_dist.cpu().numpy()[rows])


def dump_test_outputs(path, z, r, asdef, cwz, calls):
    """One test batch's results (what a result npz stores per sample) as float64 .npy files: z-scores and ratios of a
    sample of the batch's samples, and the chromosome-wide z-scores, sigma averages and calls (sample, chromosome,
    start bin, end bin, z) of all of them."""
    b, n = z.shape
    samples = _sample_rows(b, max(1, DUMP_TEST_BYTES // (16 * n)))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "test_z.npy"), z.cpu().numpy()[samples])
    np.save(os.path.join(path, "test_r.npy"), r.cpu().numpy()[samples])
    np.save(os.path.join(path, "test_asdef.npy"), asdef.cpu().numpy().astype(np.float64))
    np.save(os.path.join(path, "test_cwz.npy"), cwz.cpu().numpy().astype(np.float64))
    np.save(os.path.join(path, "test_calls.npy"),
            np.stack([calls[f].astype(np.float64) for f in ("sample", "chrom", "x", "y", "z")], axis=1).reshape(-1, 5))


def fp64_peak():
    path = os.path.join(ROOT, "profiles", "fp64_peak_r01.json")
    try:
        with open(path) as fh:
            d = json.load(fh)
        return float(d["fp64_peak_tflops"]), float(d["fp64_sustained_tflops"]), "profiles/fp64_peak_r01.json"
    except Exception:
        return 37.2, 37.2, "nominal 148 SM x 64 FMA/clk x 1.965 GHz (no measured file)"


# --------------------------------------------------------------------------------------------------------
# clocks sampler
# --------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    FIELDS = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active," \
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s, p in zip(sm, power) if p > 250.0] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------------------
# CPU reference arm
# --------------------------------------------------------------------------------------------------------
def _ref_part_worker(args):
    """One part of the reference's own getReference, in a worker process (wisecondor.py:47-56 runs parts in a
    ProcessPoolExecutor the same way)."""
    path, bins, k, part, parts = args
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        import wisetools as ref_wisetools
        X = np.load(path, mmap_mode="r")
        X = np.asfortranarray(X)            # the layout the reference's arrays have after the prep-npz round trip
        sums = list(np.cumsum(bins))
        t0 = time.time()
        idx, dist = ref_wisetools.getReference(X, bins, sums, k, part, parts)
        dt = time.time() - t0
    return idx.shape[0], dt


def cpu_reference_run(X, bins, k, steps, warmup, rows_per_core=None, budget_s=20.0):
    """Times the reference CPU path on all host cores on a bounded slice of target rows.
    Returns (pairs_per_s, dict describing the run)."""
    cores = os.cpu_count() or 1
    n = int(sum(bins))
    S = X.shape[1]
    have_ref = os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "wisetools.py"))
    if have_ref:
        import concurrent.futures
        import tempfile
        # per-row cost of the numpy path ~ 4.6e-9 s per (candidate, sample) element on one core
        est_row_s = 4.6e-9 * n * S + 2.2e-6 * n
        if rows_per_core is None:
            rows_per_core = int(max(1, min(64, budget_s / max(1, steps + warmup) / est_row_s)))
        parts = max(cores, n // rows_per_core)
        tmp = tempfile.NamedTemporaryFile(suffix=".npy", delete=False)
        tmp.close()
        np.save(tmp.name, X)
        times = []
        pairs = 0
        try:
            with concurrent.futures.ProcessPoolExecutor(max_workers=cores) as ex:
                for it in range(warmup + steps):
                    first = 1 + (it * cores) % max(1, parts - cores)
                    jobs = [(tmp.name, list(bins), k, p, parts) for p in range(first, first + cores)]
                    res = list(ex.map(_ref_part_worker, jobs))
                    dt = max(r[1] for r in res)      # parts run concurrently: the step lasts as long as the slowest
                    if it >= warmup:
                        times.append(dt)
                        pr = 0
                        for p in range(first, first + cores):
                            a, b = get_part(p - 1, parts, n)
                            pr += pairs_for_rows(bins, a, b)
                        pairs += pr
        finally:
            os.unlink(tmp.name)
        total = float(sum(times))
        desc = {"kind": "reference", "cores": cores,
                "sample": "oracle/_ref wisetools.getReference, %d parts of %d (about %d target rows each) per step on "
                          "%d worker processes, %d steps; whole-matrix candidates, S=%d" %
                          (cores, parts, n // parts, cores, steps, S)}
        return pairs / total, total / max(1, steps), desc
    # C port of the oracle (pthreads, all cores)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    est_row_s = 1.1e-9 * n * S
    rows = int(max(cores, min(n, budget_s / max(1, steps + warmup) / est_row_s * cores)))
    times = []
    pairs = 0
    for it in range(warmup + steps):
        r0 = (it * rows) % max(1, n - rows)
        t0 = time.time()
        c_oracle.get_reference_rows(X, bins, r0, r0 + rows, k, cores)
        dt = time.time() - t0
        if it >= warmup:
            times.append(dt)
            pairs += pairs_for_rows(bins, r0, r0 + rows)
    total = float(sum(times))
    desc = {"kind": "port", "cores": cores,
            "sample": "oracle/wc_oracle.c (C port, pthreads) on %d target rows per step, %d steps; oracle/_ref absent" %
                      (rows, steps)}
    return pairs / total, total / max(1, steps), desc


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    binsize, S, k, cfg = WORKLOADS[args.workload]
    bins = synth.chrom_bins(binsize)
    X = synth.corrected_like(bins, S, seed=4)
    value, s_per_step, desc = cpu_reference_run(X, bins, k, max(1, args.steps), max(0, args.warmup),
                                                budget_s=args.cpu_budget * 4)
    desc = dict(desc)
    desc["value"] = value
    desc["unit"] = UNIT
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "baseline_config": cfg, "bins": int(sum(bins)), "samples": S,
                   "refsize": k, "note": "each step is a bounded slice of target rows; throughput is per bin pair"},
        "cpu_baseline": desc,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------------------
# test half of the path: samples/s of the batched z-score + segmentation kernels (sample-sharded, no communication)
# --------------------------------------------------------------------------------------------------------
def synthetic_test_counts(nsamples, nraw, seed):
    """Per-sample raw count vectors [B][Nraw] int32: Poisson around a shared bin profile with one aberrant stretch."""
    rng = np.random.default_rng(seed)
    lam = rng.gamma(20.0, 8.7, size=nraw)
    out = rng.poisson(lam, size=(nsamples, nraw)).astype(np.int32)
    for b in range(nsamples):
        a = int(rng.integers(0, nraw - 500))
        w = int(rng.integers(20, 400))
        out[b, a:a + w] = (out[b, a:a + w] * rng.choice([0.8, 1.25])).astype(np.int32)
    return out


def cpu_reference_test(bins, idx_h, dist_h, cutoff, thr, budget_s=15.0):
    """The reference's own test path on ONE host core (it has no multi-CPU option for `test`; run.sh loops over samples):
    repeatTest on one synthetic sample, and fillTri + segmentTri on one small chromosome, extrapolated to all
    chromosomes by triangle entries (the reference's cost is per entry).  Returns (samples/s, description)."""
    import contextlib
    import io
    n = int(sum(bins))
    sums = [int(v) for v in np.cumsum(bins)]
    rng = np.random.default_rng(7)
    test = 1.0 + rng.normal(0, 0.03, size=n)
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    have_ref = os.path.isfile(os.path.join(ref_dir, "wisetools.py"))
    sys.path.insert(0, ref_dir if have_ref else os.path.join(ROOT, "oracle"))
    with contextlib.redirect_stdout(io.StringIO()):
        if have_ref:
            import wisetools as ref_wt
            t0 = time.time()
            z, r, sizes, sd = ref_wt.repeatTest(np.copy(test), idx_h, dist_h, bins, sums, cutoff, thr, 5)
            tz = time.time() - t0
        else:
            import wc_oracle
            t0 = time.time()
            z, r, sizes, sd = wc_oracle.repeat_test(np.copy(test), idx_h, dist_h, bins, sums, cutoff, thr, 5)
            tz = time.time() - t0
        # smallest chromosome whose triangle still takes a measurable time; cost model: seconds per triangle entry
        c = int(np.argmin(bins))
        zc = z[sums[c] - bins[c]:sums[c]]
        zc = zc[np.isfinite(zc)][:max(50, int((budget_s * 2 / 6e-6) ** 0.5))]
        t0 = time.time()
        if have_ref:
            ref_wt.fillTri(zc).segmentTri(thr, 3)
        else:
            wc_oracle.segment_region(zc, thr, 3)
        tseg = time.time() - t0
    entries_c = len(zc) * (len(zc) + 1) / 2.0
    entries_all = float(sum(b * (b + 1) // 2 for b in bins))
    tseg_all = tseg * entries_all / entries_c
    desc = {"kind": "reference" if have_ref else "port", "cores": 1, "unit": "samples/s",
            "zscore_s_per_sample": tz, "segmentation_s_per_sample_extrapolated": tseg_all,
            "sample": "%s repeatTest (5 passes) on 1 sample, %d bins: %.1f s; fillTri + segmentTri on %d bins of the smallest "
                      "chromosome: %.2f s for %.3g triangle entries, extrapolated to the %.3g entries of all chromosomes; one "
                      "host core (the reference tests samples one by one)" %
                      ("oracle/_ref wisetools" if have_ref else "oracle/wc_oracle.py", n, tz, len(zc), tseg, entries_c, entries_all)}
    desc["value"] = 1.0 / (tz + tseg_all)
    return desc


def bench_test_path(args, torch, dist, device, dev, rank, world, local, X, bins, k, idx_full, dist_full):
    n = int(sum(bins))
    B = int(args.test_batch)
    dist_h = dist_full.cpu().numpy()
    cut = float("inf")
    for _ in range(3):                              # getOptimalCutoff (wisetools.py:328-336), once per reference
        sel = dist_h[dist_h < cut]
        cut = np.average(sel) + 3 * np.std(sel)
    table = device.ReferenceTable(idx_full.cpu().numpy(), dist_h, bins, cut, device=local)
    counts_pinned = torch.from_numpy(synthetic_test_counts(B, n, seed=100 + rank)).pin_memory()
    masked_raw = torch.arange(n, dtype=torch.int32, device=dev)          # synthetic reference: nothing masked out
    mean = X.mean(dim=1) / X.mean(dim=1).sum()                            # a plausible pca_mean (normalised profile)
    comps = torch.zeros((3, n), dtype=torch.float64, device=dev)
    comps[0, 0::3] = 1.0
    comps[1, 1::3] = 1.0
    comps[2, 2::3] = 1.0
    comps /= comps.norm(dim=1, keepdim=True)
    thr = 5.4                                                             # norm.ppf(1 - 1/(57633*0.5*1000))
    host_z = torch.empty((B, n), dtype=torch.float64).pin_memory()
    host_r = torch.empty((B, n), dtype=torch.float64).pin_memory()
    host_n = torch.empty((B, n), dtype=torch.int32).pin_memory()

    copy_out = torch.cuda.Stream(device=dev)
    last = {}               # --dump-outputs: the results of the latest batch
    in_flight = []          # (device tensors, copy-finished event) of the batches whose results are still travelling

    host_cwz = torch.empty((B, 22), dtype=torch.float64).pin_memory()
    host_sd = torch.empty((B,), dtype=torch.float64).pin_memory()

    def run(from_host, full=False):
        counts = counts_pinned.to(dev, non_blocking=True) if from_host else counts_dev
        T = device.test_prep(counts, masked_raw, mean, comps)
        z, r, sizes, asdef = device.zscore_batch(T, B, table, thr, 5)
        cwz, cleaned, calls = device.segment_batch(z, sizes, bins, list(range(22)), 25, thr, 3)   # calls: on the host already
        if args.dump_outputs:
            last.update(z=z, r=r, asdef=asdef, cwz=cwz, calls=calls)
        if from_host and not full:      # compact result: calls, chromosome-wide z, sigma average (what a report needs)
            host_cwz.copy_(torch.as_tensor(cwz).reshape(B, -1)[:, :22], non_blocking=True)
            host_sd.copy_(torch.as_tensor(asdef).reshape(-1)[:B], non_blocking=True)
        if from_host and full:  # also the per-bin vectors, on a second stream while the next batch computes
            ready = torch.cuda.Event()
            ready.record(torch.cuda.current_stream(dev))
            with torch.cuda.stream(copy_out):
                copy_out.wait_event(ready)
                host_z.copy_(z, non_blocking=True)
                host_r.copy_(r, non_blocking=True)
                host_n.copy_(sizes, non_blocking=True)
                done = torch.cuda.Event()
                done.record(copy_out)
            in_flight.append(((z, r, sizes), done))     # keep the device buffers alive until their copy has finished
            while len(in_flight) > 1:
                in_flight.pop(0)[1].synchronize()
        return len(calls)

    counts_dev = counts_pinned.to(dev)
    for _ in range(2):
        ncalls = run(False)
    torch.cuda.synchronize(dev)
    steps = args.steps
    zs, sg, pr, executed = [], [], [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(steps):
        run(False)
        st = device.last_test_stats(local)
        zs.append(st["zscore_ms"]); sg.append(st["segment_ms"]); pr.append(st["prep_ms"])
        executed.append(st["zscore_pairs_per_pass"])
    e1.record()
    torch.cuda.synchronize(dev)
    if args.dump_outputs and rank == 0:
        dump_test_outputs(args.dump_outputs, **last)
    dev_ms = e0.elapsed_time(e1) / steps
    e2e_steps = steps
    e2e_both = []
    for full in (False, True):
        run(True, full)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        t0 = time.time()
        for _ in range(e2e_steps):
            run(True, full)
        torch.cuda.synchronize(dev)           # includes the last batch's device-to-host copies
        e2e_both.append((time.time() - t0) / e2e_steps)
    t = torch.tensor([dev_ms] + e2e_both, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_s, e2e_full_s = float(t[0].item()), float(t[1].item()), float(t[2].item())
    if rank != 0:
        return None
    zms, sms = float(np.mean(zs)), float(np.mean(sg))
    # gathered operand bytes actually executed: every pass's computed (bin, sample) pairs x mean kept refs x 8 B, twice
    # (mean pass and sum-of-squares pass); later passes only recompute what a newly marked bin can change
    mean_refs = float(table.count.float().mean().item())
    pairs_per_pass = [float(np.mean([e[p] for e in executed])) for p in range(len(executed[0]))]
    gathers = 2.0 * sum(pairs_per_pass) * mean_refs * 8.0
    entries = float(sum(b * (b + 1) // 2 for b in bins)) * B              # run evaluations (upper bound: no bin dropped)
    hbm = None
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            hbm = float(json.load(fh)["hbm_gbs"])
    except Exception:
        pass
    l2_peak = None
    try:
        with open(os.path.join(ROOT, "profiles", "l2_peak_r03.json")) as fh:
            l2_peak = float(json.loads(fh.readline())["ldg128_gbs"])
    except Exception:
        pass
    props = torch.cuda.get_device_properties(dev)
    issue_peak = props.multi_processor_count * 4 * 32 * 1.965e9
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_test(bins, idx_full.cpu().numpy(), dist_h, cut, thr)
    return {
        "cpu_baseline": cpu,
        "metric": "test_samples_per_s", "value": world * B / (dev_ms * 1e-3), "unit": "samples/s",
        "samples_per_gpu": B, "n_gpus": world, "bins": n, "refsize": k, "repeats": 5, "ms_per_batch": dev_ms,
        "phases_ms": {"prep": float(np.mean(pr)), "zscore": zms, "segment": sms}, "calls_in_batch": ncalls,
        "zscore_gather_gbs": gathers / (zms * 1e-3) / 1e9, "hbm_peak_gbs_measured": hbm,
        "zscore_pairs_per_pass": pairs_per_pass,
        "zscore_note": "executed gathers (computed pairs per pass x kept refs x 8 B x 2 reductions) per second of the "
                       "whole z-score phase (marks, work lists, sigma average and transposes included); operands come "
                       "from L2, not HBM",
        "segment_run_evals_per_s": entries / (sms * 1e-3),
        "roofline": {
            "K8": {"bound": "l2", "achieved": gathers / (zms * 1e-3) / 1e9, "peak": l2_peak, "unit": "GB/s",
                   "frac": (gathers / (zms * 1e-3) / 1e9 / l2_peak) if l2_peak else None,
                   "note": "executed gather bytes of the whole z-score phase against the L2 -> SM figure of tools/l2_peak.cu "
                           "(profiles/l2_peak_r03.json); the working copy of a 32-sample tile (15 MB) is L2-resident"},
            "K9": {"bound": "issue", "achieved": entries / (sms * 1e-3), "peak": issue_peak / 2.4, "unit": "run evaluations/s",
                   "frac": entries / (sms * 1e-3) / (issue_peak / 2.4),
                   "note": "fp32 sweep: FADD + FMNMX(|.|) per run evaluation and two shared-memory loads per five of them "
                           "(the 1/sqrt(length) multiply once per length); ceiling = SMs x 4 schedulers x 32 lanes x max SM "
                           "clock / 2.4 instructions; the whole segmentation phase (exact re-scores, recursion) is in the time"}},
        "e2e": {"value": world * B / e2e_s, "unit": "samples/s", "h2d_bytes_per_step": B * n * 4,
                "d2h_bytes_per_step": B * (22 + 1) * 8 + ncalls * 24,
                "api": "device.test_prep + zscore_batch + segment_batch from pinned host counts; calls, chromosome-wide z and "
                       "sigma averages back (the compact result a report needs), %d batches" % e2e_steps},
        "e2e_full": {"value": world * B / e2e_full_s, "unit": "samples/s", "h2d_bytes_per_step": B * n * 4,
                     "d2h_bytes_per_step": B * n * 20 + B * (22 + 1) * 8 + ncalls * 24,
                     "api": "as e2e, plus the per-bin z, ratio and refsize vectors of every sample copied back to pinned host "
                            "memory on a second stream overlapping the next batch (what a result npz holds)"},
        "parallelism": "samples sharded over %d GPU(s), no communication" % world,
    }



def parity_check(device, torch, X, X_host_np, bins, k, table_idx, table_dist, rank, world, local, rows_per=None, rows_per_range=32):
    """After the timed region: the table the timed code path produced against (a) the C restatement of the oracle on
    sampled row ranges (random ones, and ranges straddling the shard boundaries) and (b) at N > 1 the whole table of a
    single-GPU search on rank 0.  TEST INFRASTRUCTURE use of oracle/ - the checker, never the thing measured."""
    if rank != 0:
        return None
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    n = int(sum(bins))
    rng = np.random.default_rng(11)
    heavy = float(n) * X.shape[1] > 2e8          # the 2000 x 10 kb matrix: an oracle row costs 1.7 Gflop - fewer, shorter ranges
    if heavy:
        rows_per_range = 8
    starts = [int(v) for v in rng.integers(0, n - rows_per_range, size=2 if heavy else 4)]
    if world > 1 and rows_per:
        for r in range(1, world):           # straddle the boundary between the bins of rank r-1 and rank r
            b = min(n - rows_per_range, max(0, r * rows_per - rows_per_range // 2))
            if len(starts) < (4 if heavy else 8):
                starts.append(int(b))
    ti, td = table_idx.cpu().numpy(), table_dist.cpu().numpy()
    Xh = X_host_np if X_host_np is not None else X.cpu().numpy()
    ranges, ok_all = [], True
    t0 = time.time()
    for r0 in sorted(set(starts)):
        oi, od = c_oracle.get_reference_rows(Xh, bins, r0, r0 + rows_per_range, k)
        ok = bool(np.array_equal(ti[r0:r0 + rows_per_range], oi) and np.array_equal(td[r0:r0 + rows_per_range], od))
        ranges.append({"row0": r0, "rows": rows_per_range, "identical": ok})
        ok_all = ok_all and ok
    out = {"oracle": "oracle/wc_oracle.c (C restatement, bit-exact compare of indexes and distances)",
           "rows_checked": rows_per_range * len(ranges), "ranges": ranges, "identical": ok_all,
           "oracle_s": time.time() - t0}
    if world > 1:
        si, sd = device.newref_topk(X, bins, 0, n, k)
        out["whole_table_equals_single_gpu_search"] = bool(torch.equal(si, table_idx) and torch.equal(sd, table_dist))
    import hashlib
    out["table_sha256"] = hashlib.sha256(ti.tobytes() + td.tobytes()).hexdigest()[:16]
    return out

# --------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------
def symmetric_shards_agree(dev, rank, world):
    """One sharded symmetric search of a small matrix on all ranks, compared with the single-GPU search of the same
    matrix (itself parity-tested against the oracle): every rank votes, the verdict is unanimous or 'no'."""
    import torch
    import torch.distributed as dist
    from wisecondor_b200 import device, shard, synth
    ok, note = 1, "agreed on every rank"
    try:
        tb = [int(b) for b in np.array(synth.chrom_bins(250000)) // 2]
        tx = torch.as_tensor(synth.corrected_like(tb, 32, seed=9), device=dev)
        tn = int(tx.shape[0])
        trial = shard.SymmetricShardedSearch(tn, 50, rank, world, dev)
        trial.run(tx, tb)
        gi, gd = trial.gather()
        pi, pd = device.newref_topk(tx, tb, 0, tn, 50)
        if not (torch.equal(gi, pi) and torch.equal(gd, pd)):
            ok, note = 0, "rank %d: sharded result differs from the single-GPU search" % rank
    except Exception as exc:          # noqa: BLE001 - any failure means: do not use it
        ok, note = 0, "rank %d: %s: %s" % (rank, type(exc).__name__, exc)
        sys.stderr.write("symmetric sharded search disabled: %s\n" % note)
    vote = torch.tensor([ok], dtype=torch.int32, device=dev)
    dist.all_reduce(vote, op=dist.ReduceOp.MIN)
    agreed = bool(int(vote.item()))
    if not agreed and ok:
        note = "another rank disagreed"
    return agreed, note


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU-baseline work in the default run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-test", action="store_true", help="skip the batched test (z-score + segmentation) section")
    ap.add_argument("--shard", default="rows", choices=["rows", "sym"],
                    help="N > 1: getPart row shards + all-gather (default), or the sharded symmetric search")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the sampled-row comparison with the C oracle")
    ap.add_argument("--test-batch", type=int, default=512, help="test samples per GPU in the test section")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as float64 .npy files: the reference-bin table "
                         "(DIR/indexes.npy, DIR/distances.npy) and the test section's batch (DIR/test_*.npy); larger outputs "
                         "keep a fixed seeded sample of rows, under 64 MB in all (bench_outputs/ is git-ignored)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from wisecondor_b200 import device

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    binsize, S, k, cfg = WORKLOADS[args.workload]
    bins = synth.chrom_bins(binsize)
    n = int(sum(bins))
    big = n * S * 8 > (1 << 31)          # the 2000 x 10 kb matrix (4.6 GB): generated on the device, no host copy
    if big:
        X = synth.corrected_like_device(bins, S, seed=4, device=dev)
        X_host_np = X_pinned = None
        args.no_test = args.no_cpu_baseline = True
    else:
        X_host_np = synth.corrected_like(bins, S, seed=4)
        X_pinned = torch.from_numpy(X_host_np).pin_memory()
        X = X_pinned.to(dev, non_blocking=False)
    from wisecondor_b200 import shard
    r0, r1 = shard.row_shard(rank, world, n)        # = the reference's getPart(rank, world, N)
    rows = r1 - r0
    rows_max = shard.max_shard_rows(world, n)
    if world > 1:
        # the rows' all-gather is one NCCL collective over a packed (indexes | distances) block; the search writes into it
        scratch = shard.RowGather(n, k, world, dev)
        out_idx, out_dist = scratch.idx_local, scratch.dist_local
        full_idx = torch.empty((n, k), dtype=torch.int32, device=dev)
        full_dist = torch.empty((n, k), dtype=torch.float64, device=dev)
    else:
        out_idx = torch.empty((rows_max, k), dtype=torch.int32, device=dev)
        out_dist = torch.empty((rows_max, k), dtype=torch.float64, device=dev)
    flush = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.int32, device=dev)   # 512 MiB > 126 MB L2

    # N > 1: the block pairs of the symmetric search divided over the ranks (shard.SymmetricShardedSearch), if a trial run
    # on a small matrix agrees with the single-GPU search on every rank; otherwise the reference's getPart row shards.
    # Default at N > 1: the reference's own partition - getPart row shards (wisetools.py:358-361), every GPU holding the whole
    # matrix, one NCCL all-gather of the rows.  --shard sym divides the symmetric search's block pairs instead (half the
    # tensor work per rank, but three more collectives per step).
    sym_search, sym_note = None, None
    if world > 1 and args.shard == "sym":
        agreed, sym_note = symmetric_shards_agree(dev, rank, world)
        if agreed:
            sym_search = shard.SymmetricShardedSearch(n, k, rank, world, dev)
            r0, r1 = sym_search.row0, max(sym_search.row0, sym_search.row1)
            rows = r1 - r0

    timing = {"on": False}

    def step():
        if sym_search is not None:
            sym_search.run(X, bins)      # threshold all-reduce + candidate all-to-all inside
            sym_search.gather()          # NCCL all-gather: every rank ends with the whole table
            return
        device.newref_topk(X, bins, r0, r1, k, out_idx[:rows], out_dist[:rows])
        if world > 1:       # NCCL all-gather of the row shards over NVLink: every rank ends with the whole table
            if timing["on"]:
                ag_ev[0].record()
            shard.allgather_rows(out_idx[:rows], out_dist[:rows], n, out_idx=full_idx, out_dist=full_dist, scratch=scratch)
            if timing["on"]:
                ag_ev[1].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(3, args.warmup) if not big else max(1, args.warmup)):
        step()
    barrier()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    k5_ms, k4_ms, k6_ms, launches = [], [], [], 0
    k5a_ms, work_ratio, filt = [], 1.0, 0
    k6c_ms, shortlisted, ag_ms = [], 0, []
    ag_ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    barrier()
    t_wall0 = time.time()
    for i in range(args.steps):
        flush.fill_(i)                       # L2 flush between timed iterations (outside the event pairs)
        timing["on"] = True
        ev[i][0].record()
        step()
        ev[i][1].record()
        timing["on"] = False
        st = device.last_search_stats(local)
        k6c_ms.append(st.get("finalize_rescore_ms", 0.0))
        shortlisted = int(st.get("k6_shortlisted", 0))
        if world > 1 and sym_search is None:
            ag_ev[1].synchronize()
            ag_ms.append(ag_ev[0].elapsed_time(ag_ev[1]))
        k4_ms.append(st["center_norms_ms"])
        k5_ms.append(st["dist_topk_ms"])
        k6_ms.append(st["finalize_ms"] + st["exhaustive_ms"])
        k5a_ms.append(st["dist_topk_first_pass_ms"])
        work_ratio = st["tiles"] / float(max(1, st["tiles_plain"]))
        filt = int(st["filter"])
        launches += int(st["launches"])
    barrier()
    t_wall = time.time() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    pairs_total = pairs_for_rows(bins, 0, n)
    value = pairs_total / (ms_per_step * 1e-3)

    # ---- end to end through the host-buffer C-ABI call --------------------------------------------------
    if big:
        e2e = None      # validation-only workload: the matrix never exists on the host
    else:
        e2e_steps = args.steps
        if world > 1:
            # every rank uploads 1/N of the matrix, NCCL all-gathers it over NVLink, searches its rows, copies them back
            sharded = shard.ShardedSearch(n, S, k, rank, world, dev, symmetric=sym_search is not None)
            sharded.run(X_pinned, bins)
            barrier()
            t0 = time.time()
            for _ in range(e2e_steps):
                hi, hd = sharded.run(X_pinned, bins)
            h2d_bytes = sharded.rows_per * S * 8
            e2e_api = "wisecondor_b200.shard.ShardedSearch.run (pinned host matrix; 1/N upload + NCCL all-gather of the matrix%s)" % (
                "; symmetric search over block pairs" if sym_search is not None else "")
        else:
            h_idx = torch.empty((rows, k), dtype=torch.int32).pin_memory().numpy()      # pinned result buffers
            h_dist = torch.empty((rows, k), dtype=torch.float64).pin_memory().numpy()
            device.newref_topk_host(X_pinned.numpy(), bins, r0, r1, k, device=local, out_idx=h_idx, out_dist=h_dist)
            barrier()
            t0 = time.time()
            for _ in range(e2e_steps):
                hi, hd = device.newref_topk_host(X_pinned.numpy(), bins, r0, r1, k, device=local, out_idx=h_idx, out_dist=h_dist)
            h2d_bytes = int(n) * S * 8
            e2e_api = "wisecondor_b200.device.newref_topk_host -> wc_newref_topk_host (pinned host buffers)"
        torch.cuda.synchronize(dev)
        e2e_s = (time.time() - t0) / e2e_steps
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
        e2e = {"value": pairs_total / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": int(rows) * k * 12, "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
               "api": e2e_api, "bytes_note": "per rank"}

    if rank == 0:
        peak, sustained, peak_src = fp64_peak()
        k5 = float(np.mean(k5_ms))
        k6 = float(np.mean(k6_ms))
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                mp = json.load(fh)
            mp_src = "MEASURED_PEAKS.json"
        except Exception:
            mp, mp_src = {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0}, "fallback of B200_PROFILING.md (no MEASURED_PEAKS.json)"
        traffic = {}
        try:      # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu --set full captures
            with open(os.path.join(ROOT, "profiles", "traffic_r03.json")) as fh:
                traffic = json.load(fh).get(args.workload if world == 1 else "", {})
        except Exception:
            pass
        # K5: SURVEY 8(d): 2*S flops per ordered bin pair of the launch's target rows.  A whole-matrix call runs the symmetric
        # search (every unordered pair of bin blocks contracted once, plus a threshold pass): work_ratio of those flops are
        # EXECUTED; achieved / frac count the executed flops, the algorithmic rate is reported next to it.
        flops = 2.0 * S * pairs_for_rows(bins, r0, r1)
        achieved = flops * work_ratio / (k5 * 1e-3) / 1e12
        burst = ms_per_step <= 50.0            # a kernel inside a long step under the power cap -> the sustained figures
        if filt == 0:
            use_peak = peak if burst else sustained
            k5_desc = ("wc_dist_topk_kernel (K5, fp64 DMMA.8x8x4 + TMA)", use_peak,
                       "measured FP64 tensor (DMMA) peak of this pool, %s (%s figure); MEASURED_PEAKS.json has no FP64 entry" %
                       (peak_src, "burst" if burst else "sustained"), "f64")
        else:
            use_peak = float(mp["bf16_tflops"] if burst else mp.get("bf16_tflops_sustained", mp["bf16_tflops"]))
            name = ("wc_dist_topk_tc_kernel (K5t: fp16 tcgen05.mma kind::f16, fp32 accumulators in TMEM, TMA operands; FILTER only - "
                    "the fp64 exact re-score of K6 decides the result)" if filt == 2 else
                    "wc_dist_topk_f16_kernel (K5h: fp16 mma.sync HMMA.16816.F32 + TMA; filter only)")
            k5_desc = (name, use_peak, "%s dense bf16/fp16 (cuBLAS, %s figure)" % (mp_src, "burst" if burst else "sustained"), "f16 -> f32")
        roof_k5 = {"bound": "tensor", "kernel": k5_desc[0], "filter_dtype": k5_desc[3],
                   "achieved": achieved, "peak": k5_desc[1], "unit": "TFLOP/s", "frac": achieved / k5_desc[1],
                   "traffic": traffic.get("k5"), "flops_per_launch": flops * work_ratio, "kernel_ms": k5,
                   "algorithmic_flops_per_launch": flops, "algorithmic_tflops": flops / (k5 * 1e-3) / 1e12,
                   "work_ratio": work_ratio, "first_pass_ms": float(np.mean(k5a_ms)),
                   "note": "kernel_ms covers every K5 launch of a step (pivot pass, threshold pass, symmetric pass); work_ratio < 1: "
                           "symmetric search, each unordered pair of bin blocks contracted once; achieved / frac count the flops issued",
                   "peak_source": k5_desc[2], "share_of_step": k5 / ms_per_step}
        # K6 = select (warp per target bin) -> K6c streaming exact re-score -> rank.  K6c is the one long kernel: every
        # shortlisted (target, candidate) pair needs the candidate's row of S doubles at the SM, strictly in sample order
        # (wisetools.py:302) - its algorithmic bytes are pairs x S x 8 (plus the target's own chunks, one per 32 pairs).
        # `traffic` (DRAM bytes, ncu) is BELOW that: the hot candidate rows are served by the L2, so the HBM fraction can
        # exceed 1 when most of the matrix fits the 126 MB L2; the L2 -> SM figure (tools/l2_peak.cu) is printed next to it.
        rows_mine = r1 - r0
        k6c = float(np.mean(k6c_ms)) if k6c_ms else 0.0
        hbm = float(mp["hbm_gbs"])
        l2_peak = None
        try:
            with open(os.path.join(ROOT, "profiles", "l2_peak_r03.json")) as fh:
                l2_peak = float(json.loads(fh.readline())["ldg128_gbs"])
        except Exception:
            pass
        if k6c > 0.0 and shortlisted > 0:
            k6_bytes = float(shortlisted) * S * 8.0 * (1.0 + 1.0 / 32.0) + float(shortlisted) * 12.0
            k6_ms_kernel = k6c
            k6_name = ("wc_fin_rescore_kernel (K6c: exact fp64 re-score in the reference's operation order; candidate rows by "
                       "cp.async.bulk into a shared-memory ring, one persistent CTA per SM)")
            k6_note = ("algorithmic bytes = re-scored (target, candidate) pairs x S x 8 B (+ the target's chunk per 32 pairs, + the "
                       "(index, distance) result); %.1f pairs per target bin for refsize %d (the fp16 filter's error window); "
                       "frac > 1 is possible: hot candidate rows come from the L2, see traffic / l2" % (shortlisted / float(max(1, rows_mine)), k))
        else:       # fused K6 (odd S, k6_split = 0)
            k6_bytes = float(rows_mine) * ((k + 1) * S * 8.0 + k * 12.0)
            k6_ms_kernel = k6
            k6_name = "wc_finalize_kernel (K6 fused: select, exact fp64 re-score in the reference's operation order, ranking)"
            k6_note = "algorithmic bytes = target bins x ((refsize + 1) rows of S doubles + refsize (index, distance) pairs)"
        k6_gbs = k6_bytes / (k6_ms_kernel * 1e-3) / 1e9
        roof_k6 = {"bound": "hbm", "kernel": k6_name,
                   "achieved": k6_gbs, "peak": hbm, "unit": "GB/s", "frac": k6_gbs / hbm,
                   "traffic": traffic.get("k6c" if k6c > 0.0 else "k6"), "bytes_per_launch": k6_bytes, "kernel_ms": k6_ms_kernel,
                   "l2": {"peak_gbs": l2_peak, "frac": (k6_gbs / l2_peak) if l2_peak else None,
                          "peak_source": "profiles/l2_peak_r03.json (tools/l2_peak.cu: 128-bit loads over an L2-resident 48 MiB buffer)"},
                   "k6_total_ms": k6, "select_and_rank_ms": (k6 - k6c) if k6c > 0.0 else None,
                   "note": k6_note, "peak_source": "%s hbm_gbs (device copy)" % mp_src, "share_of_step": k6_ms_kernel / ms_per_step}
        k6 = k6_ms_kernel if k6c > 0.0 else k6
        roofline, roof_other = (roof_k5, roof_k6) if k5 >= k6 else (roof_k6, roof_k5)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup) if not big else max(1, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "baseline_config": cfg, "bins": n, "samples": S, "refsize": k,
                       "bin_pairs": pairs_total, "parallelism": (
                           "block pairs of the symmetric search divided over %d GPUs; NCCL all-reduce(MIN) of the bins' "
                           "thresholds, all-to-all of the column-side candidates, all-gather of the rows" % world
                           if sym_search is not None else
                           "rows sharded by getPart over %d GPU(s)%s" % (world, " + NCCL all-gather" if world > 1 else "")),
                       "sharded_symmetric_trial": sym_note,
                       "l2": "512 MiB buffer written between timed iterations (L2 flush)"},
            "phases_ms": {"center_norms": float(np.mean(k4_ms)), "dist_topk": k5, "finalize": float(np.mean(k6_ms)),
                          "finalize_rescore": float(np.mean(k6c_ms)) if k6c_ms else 0.0,
                          "allgather": float(np.mean(ag_ms)) if ag_ms else 0.0,
                          "host_and_gaps": ms_per_step - float(np.mean(k4_ms)) - k5 - float(np.mean(k6_ms)) - (float(np.mean(ag_ms)) if ag_ms else 0.0)},
            "roofline": roofline, "roofline_second_kernel": roof_other, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "wall_s_timed_region": t_wall,
        }
        if world == 1 and not args.no_cpu_baseline:
            v, s_per_step, desc = cpu_reference_run(X_host_np, bins, k, 1, 0, budget_s=args.cpu_budget)
            desc = dict(desc)
            desc["value"] = v
            desc["unit"] = UNIT
            line["cpu_baseline"] = desc
        else:
            line["cpu_baseline"] = None
    # ---- parity of what the timed code path produced (after the timed region; rank 0 checks, all ranks gather) ----
    if sym_search is not None:
        table_idx, table_dist = (t.contiguous() for t in sym_search.gather())
    elif world == 1:
        table_idx, table_dist = out_idx[:rows], out_dist[:rows]
    else:
        table_idx, table_dist = full_idx, full_dist
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, table_idx, table_dist)
    pc = None
    if not args.no_parity_check:
        pc = parity_check(device, torch, X, X_host_np, bins, k, table_idx, table_dist, rank, world, local,
                          rows_per=sym_search.rows_per if sym_search is not None else rows_max)
    if rank == 0:
        line["config"]["parity_check"] = pc
    if world > 1:
        dist.barrier()
    # ---- the test half of the path (BASELINE metric "test samples/s"): batched z-scores + segmentation ----------
    test_line = None
    if not args.no_test:
        test_line = bench_test_path(args, torch, dist, device, dev, rank, world, local, X, bins, k, table_idx, table_dist)
    if rank == 0:
        line["test"] = test_line
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
