#!/usr/bin/env python
"""Time LD pruning (tdsfs_ld_prune: k_ld_pairs, then k_ld_resolve) on bench.py's config 5 and config 4 panels, built in HBM
by the same device generator, for (size, step) in (50, 5), (100, 20), (500, 50) at threshold 0.2.

  python tools/bench_ldprune.py [--calls 5] [--warmup 1] [--out DIR]

Per workload and (size, step) it reports
  * the medians (and min / max) over synchronous calls of the CUDA-event times the library records around k_ld_pairs and
    k_ld_resolve;
  * the tested pairs, computed on the host from the chromosome offsets, size and step; the 32-sample word pairs they imply
    (tested pairs x word pairs per row) and the popcounts (9 per word pair), and popcounts per second over the k_ld_pairs
    median;
  * the kept count, and the card's name and power limit read in the same process.
The synthetic rows are drawn independently, so almost nothing is pruned; the pair kernel's cost does not depend on the data,
the resolve kernel's only through the mask bits it meets.  One JSON line per measurement on stdout; with --out, also
DIR/bench_ldprune.json.
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

CASES = ((50, 5), (100, 20), (500, 50))
THRESHOLD = 0.2
NOTE = ("synthetic rows are drawn independently, so almost nothing is pruned; the pair kernel's cost does not depend on "
        "the data")


def tested_pairs(off, size, step):
    """Row pairs i < j of one chromosome that share a window [c0 + k step, c0 + k step + size)."""
    total = 0
    for a, b in zip(off[:-1], off[1:]):
        J = np.arange(int(b - a), dtype=np.int64)        # row j's offset in its chromosome
        k = np.maximum(0, (J - size) // step + 1)        # first window that holds row j
        total += int(np.maximum(0, J - k * step).sum())  # rows i from that window's start up to j - 1
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default="config5,config4")
    ap.add_argument("--out", help="directory for bench_ldprune.json")
    args = ap.parse_args()
    import torch
    import tdsfs_capi as T
    if not torch.cuda.is_available():
        raise SystemExit("bench_ldprune.py: no CUDA device (the product has no CPU path)")
    name, limit = card()
    h = T.Handle(0)
    lines = []
    for wl in args.workloads.split(","):
        cfg = dict(WORKLOADS[wl])
        n1, n2, S = cfg["n1"], cfg["n2"], cfg["S"]
        w1, w2 = words_for(n1), words_for(n2)
        off = np.concatenate([[0], np.cumsum(chrom_sizes(S, cfg["C"]))]).astype(np.int64)
        pos = np.concatenate([np.arange(1, b - a + 1) * 50 for a, b in zip(off[:-1], off[1:])]).astype(np.int32)
        h.set_panel(n1, n2, True)
        G = torch.empty(((S + 31) // 32 * (w1 + w2) * 32,), dtype=torch.int32, device="cuda:0")
        h.synth_genotypes(G.data_ptr(), S, 0, w1, w2, n1, n2, cfg["seed"])
        h.load_genotypes(G, S, w1, w2, n1, n2, torch.from_numpy(pos).cuda(), off)
        torch.cuda.synchronize()
        for size, step in CASES:
            for _ in range(args.warmup):
                h.ld_prune(size, step, THRESHOLD)
            pairs_ms, resolve_ms, kept = [], [], None
            for _ in range(args.calls):
                keep = h.ld_prune(size, step, THRESHOLD)
                t = h.timings()
                pairs_ms.append(t["ld_pairs"])
                resolve_ms.append(t["ld_resolve"])
                kept = int(keep.sum())
            npairs = tested_pairs(off, size, step)
            word_pairs = npairs * ((w1 + w2) // 2)
            pm = float(np.median(pairs_ms))
            rec = {"workload": wl, "desc": cfg["name"], "S": S, "n1": n1, "n2": n2, "chromosomes": cfg["C"], "size": size,
                   "step": step, "threshold": THRESHOLD, "calls": args.calls,
                   "ld_pairs_ms_median": pm, "ld_pairs_ms_min": float(np.min(pairs_ms)), "ld_pairs_ms_max": float(np.max(pairs_ms)),
                   "ld_resolve_ms_median": float(np.median(resolve_ms)), "ld_resolve_ms_min": float(np.min(resolve_ms)),
                   "ld_resolve_ms_max": float(np.max(resolve_ms)),
                   "tested_pairs": npairs, "word_pairs": word_pairs, "popcounts": 9 * word_pairs,
                   "popcounts_per_s": 9 * word_pairs / (pm * 1e-3), "kept": kept, "pruned": S - kept,
                   "card": name, "power_limit": limit, "note": NOTE}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        del G
        torch.cuda.empty_cache()
    h.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_ldprune.json"), "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
