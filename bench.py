#!/usr/bin/env python
"""Benchmark of the 2D-SFS + T2D/T1D window scan (BASELINE.json metric: SNPs/s, % of HBM roofline).

  python bench.py [--gpus N --steps K --warmup W]                 our CUDA path (libtdsfs.so through the C ABI)
  python bench.py --impl reference [--gpus N --steps K --warmup W] the reference's CPU algorithm (oracle port) on host cores
  python bench.py ... --dump-outputs DIR                          also writes the window table of the last timed step to DIR

One step = one pass of the hot path over the whole workload: genotype matrix + positions -> per-SNP counts/keys and
genome-wide background spectra -> (all-reduce of the background across GPUs) -> window boundaries -> per-window
T2D / T1D(pop1) / T1D(pop2).  `value` times it with the inputs resident in HBM; `e2e` times the same pass through the
C-ABI call with pinned HOST buffers (host->device copy of the genotype matrix + positions and device->host read of
the window results inside the timed region).  Workload: BASELINE.json configs[4] (50 M SNPs x 2 pops x 500 diploids,
20 kb windows) -- the configuration the metric's target is quoted on; it fits one B200 (12.8 GB), and at N > 1 it is
sharded by contiguous chromosome ranges (total work fixed: "scaling": "strong").
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "2dsfs-scan_b200")
if PKG not in sys.path:
    sys.path.insert(0, PKG)

WORKLOADS = {
    # BASELINE.json configs[4] / SURVEY.md 8(d) row 5
    "config5": dict(S=50_000_000, n1=500, n2=500, C=32, W=20000, seed=20241005, mean_gap=50,
                    name="synthetic 50M SNPs x 2 pops x 500 diploids, 20 kb windows, genome-wide background"),
    # BASELINE.json configs[3] / SURVEY.md 8(d) row 4
    "config4": dict(S=10_000_000, n1=200, n2=200, C=32, W=20000, seed=20241004, mean_gap=50,
                    name="synthetic 10M SNPs x 2 pops x 200 diploids, 20 kb windows, genome-wide background"),
    "tiny": dict(S=400_000, n1=200, n2=200, C=8, W=20000, seed=7, mean_gap=50, name="tiny smoke workload"),
}


def words_for(n):
    """uint32 words per SNP of one population: a (lo plane, hi plane) pair per 32 samples (tdsfs_pack.words_for)"""
    return 2 * max(1, (n + 31) // 32)


def chrom_sizes(S, C):
    base = S // C
    return [base + (1 if i < S - base * C else 0) for i in range(C)]


def positions_for(cfg, chroms):
    """cumsum of Geometric(1/mean_gap) gaps from 1, seeded per chromosome (identical for any sharding)."""
    sizes = chrom_sizes(cfg["S"], cfg["C"])
    out = []
    for c in chroms:
        rng = np.random.default_rng(cfg["seed"] * 1000 + c)
        out.append(np.cumsum(rng.geometric(1.0 / cfg["mean_gap"], size=sizes[c]), dtype=np.int64).astype(np.int32))
    return out


def shard_chroms(C, world, rank):
    """contiguous chromosome ranges, balanced by SNP count (equal-size chromosomes here)"""
    lo, hi = C * rank // world, C * (rank + 1) // world
    return list(range(lo, hi))


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    def __init__(self, index):
        self.index, self.samples, self._stop, self.th = index, [], threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:  # noqa: BLE001
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.dev, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.dev)
                except Exception:  # noqa: BLE001
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.dev)
                pw = nv.nvmlDeviceGetPowerUsage(self.dev) / 1000.0
                self.samples.append((time.time(), sm, rs, pw))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.02)

    def start(self):
        if self.nv:
            self.th = threading.Thread(target=self._run, daemon=True)
            self.th.start()

    def stop(self):
        self._stop.set()
        if self.th:
            self.th.join(timeout=1)

    def summary(self, windows):
        if not self.nv or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        nv = self.nv
        sel = [s for s in self.samples if any(a <= s[0] <= b for a, b in windows)] or self.samples
        sm = sorted(s[1] for s in sel)
        bits = 0
        for s in sel:
            bits |= s[2]
        names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4,
                 "hw_power_brake": 0x80, "sync_boost": 0x10, "applications_clocks_setting": 0x2, "display_clock_setting": 0x100}
        reasons = [k for k, v in names.items() if bits & v]
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(self.dev, nv.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            mx = None
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": reasons, "samples": len(sel),
                "power_w_max": round(max(s[3] for s in sel), 1)}


# ------------------------------------------------------------------------------------------------ CPU arms (oracle)
def numpy_panel(cfg, rows, seed):
    """Host-side synthetic panel with the distribution family of the device generator (log-uniform ancestral frequency,
    per-population drift with F = 0.05, Binomial(2, p) calls, 2 % missing), generated in chunks.  Used by the reference arm,
    which must not touch libtdsfs at all."""
    from tdsfs_pack import _pack_block, to_b32
    rng = np.random.default_rng(seed)
    n1, n2 = cfg["n1"], cfg["n2"]
    lo, hi = 1.0 / (4.0 * (n1 + n2)), 1.0 - 1.0 / (4.0 * (n1 + n2))
    out = []
    for r0 in range(0, rows, 32768):
        m = min(32768, rows - r0)
        pa = lo * np.exp(rng.random(m) * np.log(hi / lo))
        blocks = []
        for ns in (n1, n2):
            p = np.clip(pa + rng.normal(0, 1, m) * np.sqrt(0.05 * pa * (1 - pa)), 0, 1).astype(np.float32)[:, None]
            a = (rng.random((m, ns), dtype=np.float32) < p).astype(np.uint8) + (rng.random((m, ns), dtype=np.float32) < p).astype(np.uint8)
            c = np.where(a == 2, 3, a).astype(np.uint8)
            c[rng.random((m, ns), dtype=np.float32) < 0.02] = 2
            blocks.append(_pack_block(c))
        out.append(np.concatenate(blocks, axis=1))
    return to_b32(np.concatenate(out, axis=0))


def sample_panel(cfg, rows, allow_gpu=True):
    """First `rows` SNP rows of chromosome 0 of the workload: device generator when allowed and a GPU is present (identical
    bytes to the GPU arm's input), numpy otherwise.  Input generation only -- never part of a timed CPU region."""
    w1, w2 = words_for(cfg["n1"]), words_for(cfg["n2"])
    if allow_gpu:
        try:
            import torch
            if torch.cuda.is_available():
                import tdsfs_capi as T
                h = T.Handle(0)
                g = torch.empty(((rows + 31) // 32 * (w1 + w2) * 32,), dtype=torch.int32, device="cuda:0")
                h.synth_genotypes(g.data_ptr(), rows, 0, w1, w2, cfg["n1"], cfg["n2"], cfg["seed"])
                G = g.cpu().numpy().view(np.uint32)
                h.close()
                return G, "device generator"
        except Exception:  # noqa: BLE001
            pass
    return numpy_panel(cfg, rows, cfg["seed"]), "numpy generator"


def oracle_modules():
    """The only place bench.py touches oracle/: the CPU baseline / reference arm."""
    import subprocess
    opath = os.path.join(ROOT, "oracle")
    if not os.path.exists(os.path.join(opath, "libsfs_oracle.so")):
        subprocess.check_call(["make", "-s", "-C", opath])
    if opath not in sys.path:
        sys.path.insert(0, opath)
    import sfs_oracle_c
    return sfs_oracle_c


def cpu_pass(OC, G, pos, cfg, nthreads):
    """One pass of the reference algorithm on a sample: decode calls -> counts, background over the sample, windows, T."""
    w1, w2 = words_for(cfg["n1"]), words_for(cfg["n2"])
    t = time.perf_counter()
    cnt = OC.decode(G, len(pos), w1, w2, cfg["n1"], cfg["n2"], nthreads=nthreads)
    r = OC.scan(cnt, pos, [0, len(pos)], cfg["n1"], cfg["n2"], W=cfg["W"], bg="genome", nthreads=nthreads)
    return time.perf_counter() - t, len(r["start"])


def cpu_sample_rate(cfg, budget_s, nthreads, steps=1, warmup=0, allow_gpu=True):
    """Time the oracle port on a bounded sample sized (by a pilot) to ~budget_s per step.  Returns dict."""
    OC = oracle_modules()
    nthreads = nthreads or OC.max_threads()
    pos_all = positions_for(cfg, [0])[0]
    per_win = cfg["W"] // cfg["mean_gap"]
    pilot_rows = min(len(pos_all), per_win * max(2 * nthreads, 8))
    G, gen = sample_panel(cfg, pilot_rows, allow_gpu)
    t_pilot, nwin = cpu_pass(OC, G, pos_all[:pilot_rows], cfg, nthreads)
    rate = pilot_rows / t_pilot
    rows = int(min(len(pos_all), max(pilot_rows, rate * budget_s)))
    if rows != pilot_rows:
        G, gen = sample_panel(cfg, rows, allow_gpu)
    pos = pos_all[:rows]
    times = []
    for i in range(warmup + steps):
        t, nwin = cpu_pass(OC, G, pos, cfg, nthreads)
        if i >= warmup:
            times.append(t)
    t_step = float(np.mean(times))
    return dict(value=rows / t_step, unit="SNPs/s", cores=nthreads, kind="port", seconds_per_step=t_step,
                sample=f"first {rows} SNPs ({nwin} windows of {cfg['W']} bp) of chromosome 0 of the workload, background over the "
                       f"sample, all {cfg['n1']}+{cfg['n2']} diploids; C restatement of the reference algorithm "
                       f"(oracle/sfs_oracle.c, dense per-window spectra), {nthreads} threads; input from the {gen}"), rows, times


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    total_budget = 150.0
    per_step = max(2.0, total_budget / (args.steps + args.warmup + 1))
    cb, rows, times = cpu_sample_rate(cfg, per_step, 0, steps=args.steps, warmup=args.warmup, allow_gpu=False)
    line = {"impl": "reference", "metric": "SNPs/sec, 2D-SFS + T2D/T1D 20 kb window scan", "value": cb["value"], "unit": "SNPs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["seconds_per_step"] * 1e3,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
            "config": {"workload": cfg["name"], "S": cfg["S"], "n1": cfg["n1"], "n2": cfg["n2"], "window_bp": cfg["W"],
                       "note": "reference is single-process Python; this arm runs its algorithm restated in C on all host cores, "
                               "on a bounded sample (SNPs/s is per-SNP throughput of the same pass)"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "SNPs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ verification
_MIX = np.array([0x9E3779B97F4A7C15, 0xC2B2AE3D27D4EB4F, 0x165667B19E3779F9, 0x27D4EB2F165667C5, 0x85EBCA77C2B2AE63,
                 0xD6E8FEB86659FD93], dtype=np.uint64)


def result_checksums(res, chrom_global, empty_bit, none_bits):
    """Order-independent integer checksums of a rank's windows (identical for every sharding of the same workload):
    sum over non-empty windows of a 64-bit mix of (chromosome, start, snp_count, n2d, n1d_p1, n1d_p2), and of the statistics
    rounded to 1e-3 (the fp64 sums of a window run in a lane order that depends on the shard's row offset)."""
    live = (res["flags"] & empty_bit) == 0
    with np.errstate(over="ignore"):
        f = [chrom_global[live].astype(np.uint64), res["start"][live].astype(np.uint64), res["snp_count"][live].astype(np.uint64),
             res["n2d"][live].astype(np.uint64), res["n1d_p1"][live].astype(np.uint64), res["n1d_p2"][live].astype(np.uint64)]
        h = np.zeros(int(live.sum()), dtype=np.uint64)
        for v, m in zip(f, _MIX):
            h = (h ^ (v * m)) * np.uint64(0xFF51AFD7ED558CCD)
            h ^= h >> np.uint64(33)
        ints = int(h.sum(dtype=np.uint64))
    out = {"windows": int(live.sum()), "snp_count_sum": int(res["snp_count"][live].sum()), "int_checksum": ints}
    for name, bit in zip(("T2D", "T1D_p1", "T1D_p2"), none_bits):
        ok = live & ((res["flags"] & bit) == 0) & np.isfinite(res[name])
        out[name + "_milli_sum"] = int(np.floor(res[name][ok] * 1000.0 + 0.5).astype(np.int64).sum())
        out[name + "_none"] = int((live & ((res["flags"] & bit) != 0)).sum())
    return out


def oracle_window_check(h, T, G, pos_host, off, res, cfg, n_sample, seed):
    """Seeded sample of this rank's windows re-scored by the CPU oracle (oracle/sfs_oracle.c decode + the oracle's dense
    spectra and likelihood) against the GPU's (all-reduced) background.  The oracle is the CHECKER here, never measured."""
    oracle_modules()
    import sfs_oracle as O
    import sfs_oracle_c as OC
    n1, n2, W = cfg["n1"], cfg["n2"], cfg["W"]
    w1, w2 = words_for(n1), words_for(n2)
    RW = w1 + w2
    g2, g1a, g1b = h.get_background(0)
    b2 = g2.astype(np.int64).ravel()[1:-1]
    b1a, b1b = O.fold_dense(g1a.astype(np.int64))[1:-1], O.fold_dense(g1b.astype(np.int64))[1:-1]
    live = np.flatnonzero((res["flags"] & T.F_EMPTY) == 0)
    rng = np.random.default_rng(seed)
    ids = rng.choice(live, size=min(n_sample, len(live)), replace=False)
    worst, bad = 0.0, 0
    for wid in ids.tolist():
        c = int(res["chrom"][wid])
        pc = pos_host[off[c]:off[c + 1]]
        lo = int(off[c] + np.searchsorted(pc, res["start"][wid], side="left"))
        hi = int(off[c] + np.searchsorted(pc, res["end"][wid], side="right"))
        if hi - lo != int(res["snp_count"][wid]):
            bad += 1
            continue
        blk0, blk1 = lo // 32, (hi + 31) // 32
        words = G[blk0 * RW * 32:blk1 * RW * 32].cpu().numpy().view(np.uint32)
        cnt = OC.decode(words, (blk1 - blk0) * 32, w1, w2, n1, n2)[lo - blk0 * 32:hi - blk0 * 32]
        e2, e1, e1b = O.dense_spectra(cnt, n1, n2)
        for name, x, b, bit in (("T2D", e2.ravel()[1:-1], b2, T.F_T2D_NONE), ("T1D_p1", O.fold_dense(e1)[1:-1], b1a, T.F_T1D_P1_NONE),
                                ("T1D_p2", O.fold_dense(e1b)[1:-1], b1b, T.F_T1D_P2_NONE)):
            exp, none = O.clr_dense(x, b)
            if none != bool(res["flags"][wid] & bit):
                bad += 1
            elif not none:
                err = abs(res[name][wid] - exp) / max(abs(exp), 1.0) if np.isfinite(exp) else (0.0 if res[name][wid] == exp else 1.0)
                worst = max(worst, float(err))
    return {"windows_checked": int(len(ids)), "max_rel_err": worst, "mismatches": int(bad), "tolerance": 1e-9,
            "ok": bool(bad == 0 and worst <= 1e-9)}


# ------------------------------------------------------------------------------------------------ GPU arm
class _DevBuf:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False), "version": 2}


def measure_workload(args, cfg, h, T, torch, dist, dev, stream, world, rank, do_e2e, verify_windows):
    """Synthesise this rank's shard of `cfg` in HBM and measure the scan on it.  Returns a dict of measurements."""
    n1, n2, W = cfg["n1"], cfg["n2"], cfg["W"]
    w1, w2 = words_for(n1), words_for(n2)
    RW = w1 + w2
    # ---- this rank's shard: contiguous chromosomes (strong) or a full copy of the workload per rank (weak)
    chroms = shard_chroms(cfg["C"], world, rank) if args.scaling == "strong" else list(range(cfg["C"]))
    sizes_all = chrom_sizes(cfg["S"], cfg["C"])
    starts_all = np.concatenate([[0], np.cumsum(sizes_all)])
    pos_list = positions_for(cfg, chroms)
    pos_host = np.concatenate(pos_list) if pos_list else np.zeros(0, np.int32)
    S_local = int(len(pos_host))
    off = np.concatenate([[0], np.cumsum([len(p) for p in pos_list])]).astype(np.int64)
    snp0 = int(starts_all[chroms[0]]) if chroms else 0
    if args.scaling == "weak":
        snp0 += rank * cfg["S"]  # different SNPs on every rank
    S_total = cfg["S"] if args.scaling == "strong" else cfg["S"] * world

    h.set_panel(n1, n2, True)
    g_words = max((S_local + 31) // 32, 1) * RW * 32  # B32 layout: blocks of 32 SNPs, zero padded
    G = torch.empty((g_words,), dtype=torch.int32, device=dev)
    h.synth_genotypes(G.data_ptr(), S_local, snp0, w1, w2, n1, n2, cfg["seed"])
    pos_dev = torch.from_numpy(pos_host).to(dev)
    torch.cuda.synchronize()

    hist_cache = {}

    def hist_tensor():
        ptr, n, _ = h.background_device()
        if ptr not in hist_cache:
            hist_cache[ptr] = torch.as_tensor(_DevBuf(ptr, n), device=dev)
        return hist_cache[ptr]

    peer = {"on": False}

    def exchange():
        """Sum the background histogram over ranks in place: the library's peer-memory kernel, else NCCL."""
        if peer["on"]:
            h.peer_reduce_finalize()  # exchange + ln tables in one launch; finalize_background below is then a no-op
        else:
            dist.all_reduce(hist_tensor())

    use_graph = not args.no_graph

    def device_step():
        """One whole pass, enqueued on one stream with no host sync: plan (K2 on a side stream, arms the fused count kernel) +
        count kernel + (exchange of the background +) ln tables + finish kernel.  tdsfs_step_bp replays the pass as a CUDA
        graph from its third call on; with the NCCL exchange (a torch call in the middle) the pass is enqueued call by call."""
        if use_graph and (world == 1 or peer["on"]):
            h.step_bp(T.BG_GENOME, W)
            return
        h.plan(W)
        h.background(T.BG_GENOME)
        if world > 1:
            exchange()
        h.finalize_background()
        h.scan(W, fetch=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    windows = []
    # ---- (A) device-resident throughput
    h.load_genotypes(G, S_local, w1, w2, n1, n2, pos_dev, off)
    if world > 1 and args.exchange == "peer":
        from tdsfs_dist import peer_setup
        h.background(T.BG_GENOME)  # allocates the histogram that the peers map
        peer["on"] = peer_setup(h)
    h.set_sync(False)
    nwarm = max(args.warmup, 3)
    launches0 = h.launch_count()
    for _ in range(nwarm):
        device_step()
    barrier()
    launches_per_step = (h.launch_count() - launches0) // nwarm
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_a0 = time.time()
    ev0.record(stream)
    for _ in range(args.steps):
        device_step()
    ev1.record(stream)
    barrier()
    t_a1 = time.time()
    windows.append((t_a0, t_a1))
    h.check()
    outputs = None
    if args.dump_outputs:  # the window table the last timed step left on the device, as a caller of tdsfs_run_bp receives it
        outputs = h.fetch_results(h.candidates(W))
        outputs["chrom"] = outputs["chrom"] + (chroms[0] if chroms else 0)
    fused, rec_bytes = h.scan_info()
    if os.environ.get("TDSFS_TAIL_STAMPS"):  # diagnostics: phases of the count kernel's tail in the last step (SM cycles of CTA 0)
        st = h.tail_stamps()
        names = ("main loop + flush", "grid barrier", "peer barrier 1", "pull + push + fence", "peer barrier 2", "ln tables", "totals")
        d = [st[i + 1] - st[i] for i in range(7)] if st[3] else [st[1] - st[0], st[2] - st[1], 0, 0, 0, st[6] - st[2], st[7] - st[6]]
        print("[rank %d] tail stamps (us at 1965 MHz): " % rank + ", ".join("%s %.1f" % (n, c / 1965.0) for n, c in zip(names, d)),
              file=sys.stderr, flush=True)
    ms_total = ev0.elapsed_time(ev1)
    tt = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_step = float(tt.item()) / args.steps
    value = S_total / (ms_step * 1e-3)

    # ---- (B) kernel-level times (CUDA events inside the library), K synchronous steps
    h.set_sync(True)
    kt = []
    t_b0 = time.time()
    for _ in range(args.steps):
        h.plan(W)
        h.background(T.BG_GENOME)
        if world > 1:
            exchange()
            torch.cuda.synchronize()
        h.finalize_background()
        h.scan(W, fetch=False)
        kt.append(h.timings())
    windows.append((t_b0, time.time()))
    kernel_ms = {k: float(np.mean([x[k] for x in kt])) for k in kt[0]}
    n_windows = h.candidates(W)
    nw_t = torch.tensor([n_windows], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(nw_t)
    n_windows_total = int(nw_t.item())

    # ---- (V) verification of the results of this very workload (after the timed regions)
    res = h.fetch_results(n_windows)
    chrom_global = res["chrom"].astype(np.int64) + (chroms[0] if chroms else 0)
    ck = result_checksums(res, chrom_global, T.F_EMPTY, (T.F_T2D_NONE, T.F_T1D_P1_NONE, T.F_T1D_P2_NONE))
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, ck)
        tot = {k: sum(p[k] for p in parts) for k in ck}
        tot["int_checksum"] %= 1 << 64
        ck = tot
    verify = dict(ck)
    verify["snp_count_sum_equals_S"] = bool(ck["snp_count_sum"] == S_total)
    verify["note"] = ("order-independent checksums over all windows of all ranks: identical for every N on the same workload "
                      "(strong scaling); statistics rounded to 1e-3 before summing")
    if rank == 0 and verify_windows > 0:
        verify["oracle"] = oracle_window_check(h, T, G, pos_host, off, res, cfg, verify_windows, cfg["seed"])
        verify["oracle"]["what"] = ("rank 0: seeded sample of windows, rows copied back from HBM and re-scored by oracle/ (C decode + dense "
                                    "spectra + multinomial log-likelihood ratio) against the GPU's all-reduced background")

    # ---- (C) end to end through the C ABI with pinned HOST buffers
    e2e = None
    if do_e2e:
        G_host = torch.empty((g_words,), dtype=torch.int32, pin_memory=True)
        G_host.copy_(G)
        pos_pin = torch.from_numpy(pos_host).pin_memory()
        torch.cuda.synchronize()

        def e2e_step():
            h.load_genotypes(G_host, S_local, w1, w2, n1, n2, pos_pin, off)
            if world > 1:
                h.plan(W)
                h.background(T.BG_GENOME)
                exchange()
                torch.cuda.synchronize()
                h.finalize_background()
                return h.scan(W, fetch=True)
            return h.run_bp(T.BG_GENOME, W, fetch=True)

        e2e_steps = max(1, min(args.steps, args.e2e_steps))
        barrier()  # rank 0 spent seconds in the oracle check above: the exchange kernels of the others must not wait for it
        res2 = e2e_step()
        barrier()
        t_c0 = time.time()
        for _ in range(e2e_steps):
            res2 = e2e_step()
        barrier()
        t_c1 = time.time()
        windows.append((t_c0, t_c1))
        wall = (t_c1 - t_c0) / e2e_steps  # host clock around synchronous C-ABI calls (copies run on the library's copy stream)
        tw = torch.tensor([wall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        d2h = sum(v.nbytes for v in res2.values())
        same = all(np.array_equal(res2[k], res[k]) if res[k].dtype != np.float64 else
                   np.allclose(res2[k], res[k], rtol=1e-10, atol=1e-10, equal_nan=True) for k in res)
        e2e = {"value": S_total / float(tw.item()), "unit": "SNPs/s", "h2d_bytes_per_step": int(g_words * 4 + S_local * 4),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": float(tw.item()) * 1e3, "steps": e2e_steps,
               "api": "tdsfs_load_genotypes(host) + tdsfs_run_bp(host results) via ctypes",
               "results_equal_device_resident_run": bool(same),
               "note": "per-rank bytes; PCIe host->device copy of the 2-bit matrix dominates"}
    if peer["on"]:
        from tdsfs_dist import peer_teardown
        peer_teardown(h)
    del G, pos_dev
    torch.cuda.empty_cache()
    return dict(value=value, ms_step=ms_step, kernel_ms=kernel_ms, launches_per_step=int(launches_per_step), e2e=e2e, verify=verify,
                n_windows_total=n_windows_total, S_local=S_local, S_total=S_total, RW=RW, windows=windows, peer=peer["on"],
                fused=fused, rec_bytes=rec_bytes, outputs=outputs)


DUMP_BYTES = 64 << 20


def write_outputs(out_dir, res, seed, cap_bytes=DUMP_BYTES):
    """One float64 .npy per result array, so that two builds can be compared window for window.  Beyond `cap_bytes` a seeded
    sample of the windows is written; window_index.npy holds the window numbers written."""
    n = len(res["start"])
    cap = cap_bytes // (8 * (len(res) + 1))
    keep = np.arange(n) if n <= cap else np.sort(np.random.default_rng(seed).choice(n, size=cap, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "window_index.npy"), keep.astype(np.float64))
    for name, v in res.items():
        np.save(os.path.join(out_dir, name + ".npy"), v[keep].astype(np.float64))


def roofline_record(cfg, m, world, workload):
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (of fallback)"
    geno_bytes = (cfg["n1"] + cfg["n2"]) / 4.0
    k1_ms = m["kernel_ms"]["k1_count"]
    achieved = m["S_local"] * geno_bytes / (k1_ms * 1e-3) / 1e9
    traffic, traffic_note = None, "not captured with ncu for this workload / shard size"
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "k1_traffic.json")))
        ent = t.get(workload, {}).get(str(world))
        if ent:
            traffic, traffic_note = ent["bytes"], ent["source"]
    except Exception:  # noqa: BLE001
        pass
    step_ms = m["ms_step"] if world == 1 else m["kernel_ms"]["pass_total"]
    step_bytes = m["S_local"] * (geno_bytes + 4.0)
    roof = {"bound": "hbm", "kernel": "k1_fused (count kernel: counts, records, background histograms, window sums)", "achieved": achieved,
            "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": m["S_local"] * geno_bytes, "kernel_ms": k1_ms,
            "whole_step": {"algorithmic_bytes": step_bytes, "ms": step_ms, "achieved": step_bytes / (step_ms * 1e-3) / 1e9},
            "kernel_ms_all": m["kernel_ms"],
            "how": "CUDA events recorded by libtdsfs on the launching stream around each kernel, mean of K synchronous steps "
                   "run right after the timed region; K1 bytes = S*(n1+n2)/4 (2-bit calls), whole step adds 4 B/SNP positions"}
    roof["whole_step"]["frac"] = roof["whole_step"]["achieved"] / peak
    return roof


def run_side(cmd, timeout):
    """A side benchmark in its own process (its JSON lines are parsed; failures are reported, not fatal)."""
    import subprocess
    try:
        r = subprocess.run([sys.executable, "-B"] + cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
        out = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{")]
        return out if r.returncode == 0 else {"error": r.stderr[-300:], "lines": out}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def run_b200(args, cfg):
    import torch
    import torch.distributed as dist
    import tdsfs_capi as T

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ.pop("NCCL_DEBUG")  # keeps NCCL's version banner off stdout: rank 0 prints exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)
    h = T.Handle(local_rank)
    # a real (non-NULL) stream shared by torch (events, NCCL ordering) and libtdsfs
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    h.set_stream(stream.cuda_stream)

    sampler = ClockSampler(local_rank)
    sampler.start()
    m = measure_workload(args, cfg, h, T, torch, dist, dev, stream, world, rank, not args.no_e2e, args.verify_windows)
    extra = {}
    if world == 1 and args.workload == "config5" and not args.no_extra:
        # BASELINE.json configs[3] (the single-GPU HBM-roofline check) in the same driver-visible record
        cfg4 = dict(WORKLOADS["config4"])
        m4 = measure_workload(args, cfg4, h, T, torch, dist, dev, stream, 1, 0, False, 0)
        extra["config4"] = {"workload": cfg4["name"], "value": m4["value"], "unit": "SNPs/s", "ms_per_step": m4["ms_step"],
                            "steps": args.steps, "windows": m4["n_windows_total"], "gpu_launches_per_step": m4["launches_per_step"],
                            "roofline": roofline_record(cfg4, m4, 1, "config4"), "verify": m4["verify"],
                            "target": "BASELINE/SURVEY 8(d) row 4: >= 37.8 G SNPs/s (0.60 of nominal 8 TB/s on the measured-peak basis)"}
        m["windows"] += m4["windows"]
    sampler.stop()
    clocks = sampler.summary(m["windows"])
    if world == 1 and rank == 0 and args.workload == "config5" and not args.no_extra:
        # BASELINE.json configs[0..2] (latency-bound, reference-sized): measured in their own processes after the timed regions
        extra["config3_sims_batch"] = run_side(["tools/bench_sims.py", "--generations", "2", "--replicates", "100", "--oracle-replicates", "2"], 240)
        extra["config1_2_ecb"] = run_side(["tools/bench_ecb.py"], 240)
    if args.dump_outputs:
        outputs = m["outputs"]
        if world > 1:  # rank order is chromosome order: the concatenation is the table of the whole workload
            parts = [None] * world
            dist.all_gather_object(parts, outputs)
            outputs = {k: np.concatenate([p[k] for p in parts]) for k in outputs}
        if rank == 0:
            write_outputs(args.dump_outputs, outputs, cfg["seed"])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    n1, n2, W = cfg["n1"], cfg["n2"], cfg["W"]
    roof = roofline_record(cfg, m, world, args.workload)
    cb = None
    if world == 1 and not args.no_cpu:
        cb, _, _ = cpu_sample_rate(cfg, args.cpu_seconds, 0)
        cb = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}

    line = {"metric": "SNPs/sec, 2D-SFS + T2D/T1D 20 kb window scan", "value": m["value"], "unit": "SNPs/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": m["ms_step"], "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "u32 popcount/histograms + f64 likelihoods", "data": "synthetic",
            "config": {"workload": cfg["name"], "S": m["S_total"], "n1": n1, "n2": n2, "window_bp": W, "windows": m["n_windows_total"],
                       "chromosomes": cfg["C"], "sharding": f"contiguous chromosome ranges over {world} rank(s)", "background": "genome-wide"
                       + ((", all-reduced in place by the library's peer-memory kernel (CUDA IPC over NVLink, uint32 sum)" if m["peer"]
                          else ", all-reduced (NCCL, uint32 sum)") if world > 1 else ""), "row_bytes": m["RW"] * 4,
                       "scan_path": ("fused: k1_fused (window sums under the count kernel) + k3_finish" if m["fused"] else "table scorer")
                       + f", {m['rec_bytes']}-byte per-SNP records" + ("" if args.no_graph else ", pass replayed as a CUDA graph (tdsfs_step_bp)"),
                       "generator": "device generator of libtdsfs (tdsfs_synth_genotypes): counter-based mix64 hash instead of Philox, "
                                    "normal approximation of the Balding-Nichols drift instead of a Beta draw (SURVEY 8(d) names Philox + Beta); "
                                    "same shape, frequency spectrum family, F = 0.05, 2 % missing; positions = cumsum of Geometric(1/50) gaps",
                       "l2": "inputs (per-rank genotype matrix %.1f GB) larger than L2" % (m["S_local"] * m["RW"] * 4 / 1e9)},
            "roofline": roof, "cpu_baseline": cb, "e2e": m["e2e"], "verify": m["verify"], "gpu_launches": int(m["launches_per_step"] * args.steps),
            "gpu_launches_per_step": m["launches_per_step"], "clocks": clocks, "extra": extra}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config5", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: background all-reduce through the library's peer-memory kernel (default) or NCCL")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--snps", type=int, default=0, help="override the SNP count (profiling runs only; not a bench value)")
    ap.add_argument("--verify-windows", type=int, default=128, help="windows re-scored by the CPU oracle after the timed region")
    ap.add_argument("--no-graph", action="store_true", help="enqueue every pass call by call instead of replaying the captured CUDA graph")
    ap.add_argument("--no-extra", action="store_true", help="skip the config4 / config3 / ECB sub-records of the default N=1 run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the window table of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm only times a sample")
    cfg = dict(WORKLOADS[args.workload])
    if args.snps:
        cfg["S"] = args.snps
        cfg["name"] += f" [REDUCED to {args.snps} SNPs: profiling run, not a bench value]"
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_b200(args, cfg)


if __name__ == "__main__":
    main()
