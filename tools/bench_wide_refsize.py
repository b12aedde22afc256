"""Device time of wc_zscore_batch (K8 for refsize <= 512, K8w above) against refsize, on two shapes.

Workload: B = 512 samples, 5 repeats, threshold 5.4, aberrations of +-20 % over 20-400 bins per sample (so the later
passes mark and recompute real work).  Refsizes 100 and 512 run on K8, 513, 1024, 2048 and 4096 on K8w.
  250 kb: N = 11 537 (the masked-size layout of the raw 250 kb bins), the table built by c_oracle.get_reference_rows on
          a 60-sample corrected-like matrix (one search at refsize 4096; rows are ordered by distance, so refsize k is
          its first k columns).
  50 kb:  N = 57 633, a synthetic table: each bin's reference bins are distinct other-chromosome bins in a random
          stride order, all below the cutoff.  The content only changes the locality of the gathers, not the work.
Reported per point: device time of wc_zscore_batch (CUDA events, median of 3 after one warm-up call), samples/s and
the gathered bytes per second at two sweeps per computed pair (sum of count x 8 B over the pairs each pass computed,
x 2; a lane that dropped a value walks a third time, which is not counted), with the card's name and power limit.

    python tools/bench_wide_refsize.py [out.json]
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
from wisecondor_b200 import device, synth  # noqa: E402

B, REPEATS, THR = 512, 5, 5.4
KS = [100, 512, 513, 1024, 2048, 4096]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def table_250kb():
    import c_oracle
    bins = synth.chrom_bins(250000)
    X = synth.corrected_like(bins, 60, seed=4)
    idx, dst = c_oracle.get_reference_rows(X, bins, 0, int(sum(bins)), max(KS))
    return bins, idx, dst


def table_50kb(k, seed=3):
    bins = synth.chrom_bins(50000)
    n = int(sum(bins))
    rng = np.random.default_rng(seed)
    idx = np.empty((n, k), dtype=np.int32)
    starts = np.concatenate(([0], np.cumsum(bins)))
    primes = np.array([7919, 104729, 1299709, 15485863], dtype=np.int64)
    for c in range(len(bins)):
        a, b = int(starts[c]), int(starts[c + 1])
        nother = n - (b - a)
        steps = primes[rng.integers(0, len(primes), size=b - a)]
        steps[np.gcd(steps, nother) != 1] = 1
        off = rng.integers(0, nother, size=b - a)
        idx[a:b] = (off[:, None] + np.arange(k, dtype=np.int64)[None, :] * steps[:, None]) % nother
    return bins, idx, np.zeros((n, k))


def workload(n):
    rng = np.random.default_rng(1)
    host = 1.0 + rng.normal(0, 0.03, size=(n, B))
    for b in range(B):
        a = int(rng.integers(0, n - 400))
        host[a:a + int(rng.integers(20, 400)), b] *= rng.choice([0.8, 1.2])
    T = torch.ones((n, device.pad32(B)), dtype=torch.float64, device="cuda")
    T[:, :B] = torch.from_numpy(host).cuda()
    return T


def measure(shape, bins, idx, dst, cutoff, T):
    table = device.ReferenceTable(idx, dst, bins, cutoff)
    n = int(sum(bins))
    count = table.count.cpu().numpy().astype(np.int64)
    device.zscore_batch(T, B, table, THR, REPEATS)
    ms = []
    for _ in range(3):
        device.zscore_batch(T, B, table, THR, REPEATS)
        torch.cuda.synchronize()
        st = device.last_test_stats()
        ms.append(st["zscore_ms"])
    pairs = list(st["zscore_pairs_per_pass"])
    pairs[0] = n * B
    # bytes: pass 0 gathers every pair; later passes the listed pairs (mean count) or, past the limit, every pair
    gathered = sum(p * float(count.mean()) * 8 * 2 for p in pairs)
    t = float(np.median(ms))
    return {"shape": shape, "N": n, "refsize": int(idx.shape[1]), "kernel": "K8w" if idx.shape[1] > 512 else "K8",
            "mean_count": float(count.mean()), "zscore_ms": t, "zscore_ms_all": ms, "samples_per_s": B / (t * 1e-3),
            "pairs_per_pass": pairs, "gathered_GB_per_s_two_sweeps": gathered / (t * 1e-3) / 1e9}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"card": card(), "B": B, "repeats": REPEATS, "threshold": THR, "points": []}
    print(res["card"], flush=True)
    bins, idx, dst = table_250kb()
    T = workload(int(sum(bins)))
    for k in KS:
        r = measure("250kb", bins, np.ascontiguousarray(idx[:, :k]), np.ascontiguousarray(dst[:, :k]), 1e30, T)
        res["points"].append(r)
        print(json.dumps(r), flush=True)
    del T
    T = None
    for k in KS:
        bins, idx, dst = table_50kb(k)
        if T is None:
            T = workload(int(sum(bins)))
        r = measure("50kb", bins, idx, dst, 1.0, T)
        res["points"].append(r)
        print(json.dumps(r), flush=True)
        del idx, dst
    if out:
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
