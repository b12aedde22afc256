"""Device time of the reference-bin search against refsize: wc_newref_topk (k = 100, for reference) and
wc_newref_topk_wide (k = 385, 1024, 2048, 4096), on 600 samples x 250 kb (N = 11 537) and 600 x 50 kb (N = 57 633)
corrected-like matrices (synth.corrected_like), all rows.

Reported per point: end-to-end device time of the call (CUDA events around it, median of 3 after one warm-up call), the
phase times the library records (narrow: K5 filter, K6 finalize, K6b exhaustive; wide: K5w distances, K6w select +
rank), rows sent to the exhaustive fallback, entries ranked per row, the fp64 rate of the wide distance phase (3 N^2 S
operations: subtract, multiply, add per pair and sample), and the card's name and power limit read in the same run.

    python tools/bench_wide_search.py [out.json]
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from wisecondor_b200 import device, synth  # noqa: E402

S = 600
KS = [100, 385, 1024, 2048, 4096]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def measure(shape, bins, x, k):
    n = int(sum(bins))
    idx = torch.empty((n, k), dtype=torch.int32, device="cuda")
    dist = torch.empty((n, k), dtype=torch.float64, device="cuda")
    device.newref_search(x, bins, 0, n, k, out_idx=idx, out_dist=dist)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(3):
        ev0.record()
        device.newref_search(x, bins, 0, n, k, out_idx=idx, out_dist=dist)
        ev1.record()
        torch.cuda.synchronize()
        ms.append(ev0.elapsed_time(ev1))
    st = device.last_search_stats()
    wide = k > device.NARROW_REFSIZE_MAX
    r = {"shape": shape, "N": n, "S": S, "refsize": k, "entry": "wide" if wide else "narrow",
         "end_to_end_ms": float(np.median(ms)), "end_to_end_ms_all": ms}
    if wide:
        r.update({"dist_ms": st["dist_topk_ms"], "select_rank_ms": st["finalize_ms"], "exhaustive_rows": 0,
                  "ranked_per_row": k, "rows_per_chunk": int(st["tiles_plain"]),
                  "dist_fp64_tflops": 3.0 * n * n * S / (st["dist_topk_ms"] * 1e-3) / 1e12})
    else:
        r.update({"center_norms_ms": st["center_norms_ms"], "filter_ms": st["dist_topk_ms"],
                  "finalize_ms": st["finalize_ms"], "exhaustive_ms": st["exhaustive_ms"],
                  "exhaustive_rows": int(st["exhaustive_rows"]),
                  "rescored_per_row": st["k6_shortlisted"] / n if st["k6_shortlisted"] > 0 else None})
    return r


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"card": card(), "points": []}
    print(res["card"], flush=True)
    for shape, binsize in (("250kb", 250000), ("50kb", 50000)):
        bins = synth.chrom_bins(binsize)
        x = torch.from_numpy(synth.corrected_like(bins, S, seed=7)).cuda()
        for k in KS:
            r = measure(shape, bins, x, k)
            res["points"].append(r)
            print(json.dumps(r), flush=True)
        del x
    if out:
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
