#!/usr/bin/env python
"""Time the per-window LD pass (tdsfs_ld_windows_*: k_ld_windows, then k_ldw_finish) on bench.py's config 5 and config 4
panels, built in HBM by the same device generator as tools/bench_ldprune.py, over 20 kb windows and 500-SNP windows.

  python tools/bench_ld_windows.py [--calls 5] [--warmup 1] [--out DIR]

Per workload and window mode it reports
  * the median, min and max over synchronous calls of the CUDA-event time the library records around the pass's kernels
    (tdsfs_timings slot 14);
  * the row pairs the windows hold, computed on the host from the window bounds; the 32-sample word pairs they imply
    (pairs x word pairs per row) and the popcounts (9 per word pair), and popcounts per second over the median;
  * the card's name and power limit read in the same process.
Cost grows with the square of a window's rows.  The synthetic rows are drawn independently, and the pair kernel's cost does
not depend on the data.  One JSON line per measurement on stdout; with --out, also DIR/bench_ld_windows.json.
"""
import argparse
import json
import os
import sys

import numpy as np

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, os.path.join(ROOT, "2dsfs-scan_b200"), HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench import WORKLOADS, chrom_sizes, words_for  # noqa: E402
from bench_diversity import card  # noqa: E402

CASES = ((20000, False), (500, True))
GAP = 50  # bp between neighbouring rows, as in tools/bench_ldprune.py: 400 rows per 20 kb window


def window_pairs(off, size, snp_mode):
    """Row pairs i < j that share a candidate window: fixed-bp windows [1 + kW, (k+1)W] over positions GAP, 2 GAP, ...;
    fixed-SNP windows are the full chunks of `size` rows of each chromosome."""
    total = 0
    for a, b in zip(off[:-1], off[1:]):
        n = int(b - a)
        if snp_mode:
            rows = np.full(n // size, size, dtype=np.int64)
        else:
            rows = np.bincount((np.arange(1, n + 1, dtype=np.int64) * GAP - 1) // size)
        total += int((rows * (rows - 1) // 2).sum())
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default="config5,config4")
    ap.add_argument("--out", help="directory for bench_ld_windows.json")
    args = ap.parse_args()
    import torch
    import tdsfs_capi as T
    if not torch.cuda.is_available():
        raise SystemExit("bench_ld_windows.py: no CUDA device (the product has no CPU path)")
    name, limit = card()
    h = T.Handle(0)
    lines = []
    for wl in args.workloads.split(","):
        cfg = dict(WORKLOADS[wl])
        n1, n2, S = cfg["n1"], cfg["n2"], cfg["S"]
        w1, w2 = words_for(n1), words_for(n2)
        off = np.concatenate([[0], np.cumsum(chrom_sizes(S, cfg["C"]))]).astype(np.int64)
        pos = np.concatenate([np.arange(1, b - a + 1) * GAP for a, b in zip(off[:-1], off[1:])]).astype(np.int32)
        h.set_panel(n1, n2, True)
        G = torch.empty(((S + 31) // 32 * (w1 + w2) * 32,), dtype=torch.int32, device="cuda:0")
        h.synth_genotypes(G.data_ptr(), S, 0, w1, w2, n1, n2, cfg["seed"])
        h.load_genotypes(G, S, w1, w2, n1, n2, torch.from_numpy(pos).cuda(), off)
        torch.cuda.synchronize()
        for size, snp in CASES:
            for _ in range(args.warmup):
                h.ld_windows(size, snp_mode=snp)
            ms, res = [], None
            for _ in range(args.calls):
                res = h.ld_windows(size, snp_mode=snp)
                ms.append(h.ld_windows_ms())
            npairs = window_pairs(off, size, snp)
            assert int(res["n_pairs_p1"].sum()) <= npairs  # n_pairs counts the defined pairs only
            word_pairs = npairs * ((w1 + w2) // 2)
            med = float(np.median(ms))
            rec = {"workload": wl, "desc": cfg["name"], "S": S, "n1": n1, "n2": n2, "chromosomes": cfg["C"],
                   "window": size, "snp_mode": snp, "windows": int(len(res["start"])), "calls": args.calls,
                   "ld_windows_ms_median": med, "ld_windows_ms_min": float(np.min(ms)), "ld_windows_ms_max": float(np.max(ms)),
                   "pairs": npairs, "word_pairs": word_pairs, "popcounts": 9 * word_pairs,
                   "popcounts_per_s": 9 * word_pairs / (med * 1e-3),
                   "zns_p1_mean": float(np.nanmean(res["zns_p1"])), "omega_p1_defined": int(np.isfinite(res["omega_p1"]).sum()),
                   "card": name, "power_limit": limit}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        del G
        torch.cuda.empty_cache()
    h.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_ld_windows.json"), "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
