#!/usr/bin/env python
"""Time the per-window diversity pass (Hudson FST, pi, dxy: tdsfs_diversity_bp), the neutrality pass (Watterson's theta,
Tajima's D: tdsfs_neutrality_bp) and the Weir and Cockerham FST pass (tdsfs_wcfst_bp) on bench.py's config 5 and config 4
panels, built in HBM by the same device generator, over the same 20 kb windows.

  python tools/bench_diversity.py [--calls 30] [--warmup 5] [--out DIR]

Per workload it reports
  * call_ms:   diversity(fetch=False) back to back, CUDA events around the whole run / calls (window boundaries, segment list
               and its prefix sum, segment kernel, finish kernel);
  * kernel_ms: the segment + finish kernels alone (events the library records around them), mean over synchronous calls;
  * the algorithmic bytes S (n1 + n2) / 4 (2-bit calls; each read once), the achieved GB/s over kernel_ms and call_ms, and
    their fraction of 6,544 GB/s (the copy rate measured for this project on a B200) and of the 7.7 TB/s data sheet;
  * copy_gbs: a device-to-device copy of the same genotype matrix timed in the same process, read + write bytes over time;
  * the card's name and power limit, read in the same process;
  * the same call / kernel times, GB/s and fractions for the neutrality pass under neutrality_* keys (same panel, same
    windows, same algorithmic bytes), and neutrality_over_fst_kernel, the ratio of the two kernel medians;
  * the same again for the Weir and Cockerham FST pass under wcfst_* keys, with wcfst_over_fst_kernel.
One JSON line per workload on stdout; with --out, also DIR/bench_diversity.json.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "2dsfs-scan_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench import WORKLOADS, chrom_sizes, positions_for, words_for  # noqa: E402

COPY_PEAK_GBS = 6544.0   # device-to-device copy rate measured for this project on a B200
SHEET_GBS = 7700.0       # HGX B200 data sheet, one GPU


def card():
    """(name, power limit) of GPU 0, read now."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [x.strip() for x in out.split(",")[:2]]
        return name, limit
    except Exception:  # noqa: BLE001
        import torch
        return torch.cuda.get_device_name(0), "unknown"


def time_pass(entry, W, args, h, torch, stream):
    """(kernel times of synchronous calls, call time of back-to-back asynchronous calls, fetched results) of the pass
    Handle.<entry>, timed as the FST pass is."""
    run, ms = getattr(h, entry), getattr(h, entry + "_ms")
    for _ in range(args.warmup):
        run(W, fetch=False)
    kernel = []
    for _ in range(args.calls):
        run(W, fetch=False)
        kernel.append(ms())
    h.set_sync(False)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.calls):
        run(W, fetch=False)
    ev1.record(stream)
    torch.cuda.synchronize()
    h.set_sync(True)
    return kernel, ev0.elapsed_time(ev1) / args.calls, getattr(h, "fetch_" + entry)(h.candidates(W))


def measure(name, cfg, args, h, T, torch, stream):
    n1, n2, W = cfg["n1"], cfg["n2"], cfg["W"]
    w1, w2 = words_for(n1), words_for(n2)
    S = cfg["S"]
    pos = np.concatenate(positions_for(cfg, range(cfg["C"])))
    off = np.concatenate([[0], np.cumsum(chrom_sizes(S, cfg["C"]))]).astype(np.int64)
    h.set_panel(n1, n2, True)
    G = torch.empty(((S + 31) // 32 * (w1 + w2) * 32,), dtype=torch.int32, device="cuda:0")
    h.synth_genotypes(G.data_ptr(), S, 0, w1, w2, n1, n2, cfg["seed"])
    pos_dev = torch.from_numpy(pos).cuda()
    h.load_genotypes(G, S, w1, w2, n1, n2, pos_dev, off)
    torch.cuda.synchronize()

    # kernel time: synchronous calls, events recorded by the library around the segment + finish kernels
    h.set_sync(True)
    for _ in range(args.warmup):
        h.diversity(W, fetch=False)
    kernel = []
    for _ in range(args.calls):
        h.diversity(W, fetch=False)
        kernel.append(h.diversity_ms())
    # call time: asynchronous calls back to back on the handle's stream
    h.set_sync(False)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.calls):
        h.diversity(W, fetch=False)
    ev1.record(stream)
    torch.cuda.synchronize()
    call_ms = ev0.elapsed_time(ev1) / args.calls
    h.set_sync(True)
    res = h.fetch_diversity(h.candidates(W))

    # the neutrality and the Weir and Cockerham FST passes over the same windows, timed the same way
    nkernel, ncall_ms, nres = time_pass("neutrality", W, args, h, torch, stream)
    wkernel, wcall_ms, wres = time_pass("wcfst", W, args, h, torch, stream)

    # same-process reference: device-to-device copy of the genotype matrix
    dst = torch.empty_like(G)
    for _ in range(3):
        dst.copy_(G)
    ev0.record(stream)
    for _ in range(args.calls):
        dst.copy_(G)
    ev1.record(stream)
    torch.cuda.synchronize()
    copy_ms = ev0.elapsed_time(ev1) / args.calls
    copy_gbs = 2 * G.numel() * 4 / (copy_ms * 1e-3) / 1e9
    del dst

    algo = S * (n1 + n2) / 4.0
    k_ms = float(np.median(kernel))
    live = (res["flags"] & T.F_EMPTY) == 0
    out = {"workload": name, "desc": cfg["name"], "S": S, "n1": n1, "n2": n2, "window_bp": W, "windows": int(len(res["start"])),
           "calls": args.calls, "call_ms": call_ms, "kernel_ms_median": k_ms, "kernel_ms_min": float(np.min(kernel)),
           "kernel_ms_max": float(np.max(kernel)), "algorithmic_bytes": algo, "matrix_bytes": int(G.numel() * 4),
           "kernel_gbs": algo / (k_ms * 1e-3) / 1e9, "call_gbs": algo / (call_ms * 1e-3) / 1e9,
           "copy_ms": copy_ms, "copy_gbs": copy_gbs,
           "checks": {"snp_count_sum_equals_S": bool(int(res["snp_count"].sum()) == S),
                      "n_sites": int(res["n_sites"].sum()), "windows_with_fst": int(np.isfinite(res["fst"][live]).sum()),
                      "mean_fst": float(np.nanmean(res["fst"][live]))}}
    nk_ms = float(np.median(nkernel))
    nlive = (nres["flags"] & T.F_EMPTY) == 0
    out.update({"neutrality_call_ms": ncall_ms, "neutrality_kernel_ms_median": nk_ms,
                "neutrality_kernel_ms_min": float(np.min(nkernel)), "neutrality_kernel_ms_max": float(np.max(nkernel)),
                "neutrality_kernel_gbs": algo / (nk_ms * 1e-3) / 1e9, "neutrality_call_gbs": algo / (ncall_ms * 1e-3) / 1e9,
                "neutrality_over_fst_kernel": nk_ms / k_ms,
                "neutrality_checks": {"snp_count_sum_equals_S": bool(int(nres["snp_count"].sum()) == S),
                                      "n_seg_p1": int(nres["n_seg_p1"].sum()), "n_seg_p2": int(nres["n_seg_p2"].sum()),
                                      "windows_with_tajima_d_p1": int(np.isfinite(nres["tajima_d_p1"][nlive]).sum()),
                                      "mean_tajima_d_p1": float(np.nanmean(nres["tajima_d_p1"][nlive])),
                                      "mean_tajima_d_p2": float(np.nanmean(nres["tajima_d_p2"][nlive]))}})
    wk_ms = float(np.median(wkernel))
    wlive = (wres["flags"] & T.F_EMPTY) == 0
    out.update({"wcfst_call_ms": wcall_ms, "wcfst_kernel_ms_median": wk_ms,
                "wcfst_kernel_ms_min": float(np.min(wkernel)), "wcfst_kernel_ms_max": float(np.max(wkernel)),
                "wcfst_kernel_gbs": algo / (wk_ms * 1e-3) / 1e9, "wcfst_call_gbs": algo / (wcall_ms * 1e-3) / 1e9,
                "wcfst_over_fst_kernel": wk_ms / k_ms,
                "wcfst_checks": {"snp_count_sum_equals_S": bool(int(wres["snp_count"].sum()) == S),
                                 "n_sites": int(wres["n_sites"].sum()),
                                 "windows_with_fst": int(np.isfinite(wres["fst"][wlive]).sum()),
                                 "mean_fst": float(np.nanmean(wres["fst"][wlive]))}})
    for k in ("kernel", "call", "neutrality_kernel", "neutrality_call", "wcfst_kernel", "wcfst_call"):
        out[k + "_frac_of_copy_peak"] = out[k + "_gbs"] / COPY_PEAK_GBS
        out[k + "_frac_of_sheet"] = out[k + "_gbs"] / SHEET_GBS
    del G, pos_dev
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workloads", default="config5,config4")
    ap.add_argument("--out", help="directory for bench_diversity.json")
    args = ap.parse_args()
    if args.calls < 20:
        ap.error("--calls must be at least 20")
    import torch
    import tdsfs_capi as T
    if not torch.cuda.is_available():
        raise SystemExit("bench_diversity.py: no CUDA device (the product has no CPU path)")
    name, limit = card()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    h = T.Handle(0)
    h.set_stream(stream.cuda_stream)
    lines = []
    for wl in args.workloads.split(","):
        rec = measure(wl, dict(WORKLOADS[wl]), args, h, T, torch, stream)
        rec["card"], rec["power_limit"] = name, limit
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    h.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_diversity.json"), "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
