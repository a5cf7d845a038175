"""Multi-GPU plumbing: one process per GPU (torchrun), windows sharded over contiguous row ranges, and ONE collective --
a sum of the integer background histogram -- where a background spans ranks (SURVEY.md section 8e).

  * rows are split into `world` contiguous pieces balanced by SNP count; a piece boundary falls on a chromosome boundary
    when one is close enough, otherwise INSIDE a chromosome on a window boundary (the first SNP at or after 1 + k W for
    fixed-bp windows, a multiple of N rows for fixed-SNP windows), so that no window is split (make_shard_plan);
  * every rank loads its pieces as its own chromosomes (a split chromosome appears on two or more ranks);
  * genome-wide background (the north-star mode, reference usage :1970-1981): in-place all-reduce of the packed histogram --
    the library's peer-memory kernel (tdsfs_peer_*) or NCCL; single-chromosome background (scan_chooseChr*, reference
    :993-1159, :1303-1420): the owning rank(s) contribute that chromosome, every other rank an all-zero histogram, and the
    same sum broadcasts it; per-chromosome backgrounds (combined_scan :809-825, scan_perChr_bySNPs :1450-1460): no collective
    for unsplit chromosomes, a sum over the ranks holding pieces of a split one;
  * results are gathered in rank order == the reference's sorted window order, with the candidates a continuing piece
    shares with its predecessor trimmed and the first fixed-SNP label of a continuing piece patched (:1527/:1535), so that
    the gathered arrays equal the single-GPU arrays entry for entry.

torch.distributed is used for the plumbing only (NCCL on GPUs, gloo in the CPU tests); the histogram lives in libtdsfs'
device memory and is reduced in place through a zero-copy tensor view.
"""
from __future__ import annotations

import numpy as np

BG_NONE, BG_PER_CHROM, BG_GENOME, BG_CHROM = 0, 1, 2, 3  # tdsfs_capi constants (kept importable without the library)
F_EMPTY = 8
UINT32_MAX = 2 ** 32 - 1


def shard_chromosomes(sizes, world):
    """Contiguous chromosome ranges balanced by SNP count.  sizes: SNPs per chromosome (sorted chromosome order).
    Returns [(lo, hi)] per rank with lo <= hi, covering [0, C) in order (a rank may be empty when world > C)."""
    sizes = np.asarray(sizes, dtype=np.int64)
    C = len(sizes)
    total = int(sizes.sum())
    bounds = [0]
    csum = np.concatenate([[0], np.cumsum(sizes)])
    for r in range(1, world):
        target = total * r / world
        # first boundary whose prefix is >= target, but keep at least monotone boundaries
        b = int(np.searchsorted(csum, target, side="left"))
        # choose the closer of b-1 / b to the target
        if b > 0 and abs(csum[b - 1] - target) <= abs(csum[min(b, C)] - target):
            b -= 1
        bounds.append(min(max(b, bounds[-1]), C))
    bounds.append(C)
    return [(bounds[r], bounds[r + 1]) for r in range(world)]


# ------------------------------------------------------------------------------------------------ shard plan
class Piece:
    """Rows [lo, hi) (global row numbers) of chromosome `chrom`; `first` = the piece starts its chromosome."""
    __slots__ = ("chrom", "lo", "hi", "first")

    def __init__(self, chrom, lo, hi, first):
        self.chrom, self.lo, self.hi, self.first = int(chrom), int(lo), int(hi), bool(first)

    def __repr__(self):
        return f"Piece(chrom={self.chrom}, rows=[{self.lo},{self.hi}), first={self.first})"


def _snap(pos, off, c, row, W, N):
    """Largest allowed split row <= `row` inside chromosome c: the first SNP of the window that holds `row`."""
    lo = int(off[c])
    if row <= lo:
        return lo
    if N is not None:
        return lo + (row - lo) // N * N
    k = max(int(pos[row]) - 1, 0) // W                      # window index of `row` (position 0 falls in window 0)
    if k == 0:
        return lo
    return lo + int(np.searchsorted(pos[lo:int(off[c + 1])], 1 + k * W, side="left"))


def make_shard_plan(pos, off, world, W=None, N=None, tol=0.05):
    """Split the rows [0, S) into `world` contiguous runs balanced by SNP count.  pos: positions of all SNPs (host array, every
    rank holds it: 4 bytes per SNP), off: chromosome offsets.  A boundary is placed on the nearest chromosome boundary when
    that costs at most `tol` of a rank's share, else inside the chromosome on a window boundary (W bp or N SNPs).
    Returns a list (one entry per rank) of lists of Piece; a rank may be empty when there is less work than ranks."""
    assert (W is None) != (N is None), "exactly one of W (fixed-bp) and N (fixed-SNP) windows"
    off = np.asarray(off, dtype=np.int64)
    C, S = len(off) - 1, int(off[-1])
    share = S / world
    cuts = [0]
    for r in range(1, world):
        target = int(round(S * r / world))
        c = int(np.searchsorted(off, target, side="right")) - 1          # chromosome holding the target row
        c = min(max(c, 0), C - 1) if C else 0
        cand = [int(off[c]), int(off[c + 1])] if C else [0]
        best = min(cand, key=lambda b: abs(b - target))
        if abs(best - target) > tol * share and C:
            inside = _snap(pos, off, c, min(target, int(off[c + 1]) - 1), W, N)
            # the window boundary at or below the target, or the one above it if that is closer
            best = inside
        cuts.append(min(max(best, cuts[-1]), S))
    cuts.append(S)
    plan = []
    for r in range(world):
        a, b = cuts[r], cuts[r + 1]
        pieces = []
        if b > a:
            c0 = int(np.searchsorted(off, a, side="right")) - 1
            c = c0
            while c < C and int(off[c]) < b:
                lo, hi = max(a, int(off[c])), min(b, int(off[c + 1]))
                if hi > lo:
                    pieces.append(Piece(c, lo, hi, lo == int(off[c])))
                c += 1
        plan.append(pieces)
    return plan


def local_offsets(pieces):
    """chrom_off of a rank's shard: its pieces, in order, as the rank's own chromosomes."""
    return np.concatenate([[0], np.cumsum([p.hi - p.lo for p in pieces])]).astype(np.int64)


# ------------------------------------------------------------------------------------------------ background exchange
class _DevBuf:
    """__cuda_array_interface__ view of a raw device pointer (uint32 counts reinterpreted as int32 for torch)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False), "version": 2}


def background_tensor(handle, device):
    """Zero-copy torch view of the handle's packed background histogram [group][2D | 1D pop1 | 1D pop2]."""
    if hasattr(handle, "background_tensor"):  # CPU stand-ins of the gloo tests
        return handle.background_tensor()
    import torch
    ptr, n, _ = handle.background_device()
    return torch.as_tensor(_DevBuf(ptr, n), device=device)


def allreduce_background(hist, group=None):
    """Sum the background histogram over ranks, in place (counts stay exact: guarded by check_total_snps)."""
    import torch.distributed as dist
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=group)
        if hist.is_cuda:
            # NCCL runs on torch's current stream, the library on its own: the tables must not be built from a histogram
            # that is still being reduced (the caller's handle is synchronous, so the other direction is already ordered)
            import torch
            torch.cuda.current_stream(hist.device).synchronize()
    return hist


def check_total_snps(local_snps, group=None):
    """The cross-rank sum runs in uint32 bins: the total number of SNPs (an upper bound of any bin) must fit."""
    import torch.distributed as dist
    total = int(local_snps)
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        parts = [None] * dist.get_world_size(group)
        dist.all_gather_object(parts, int(local_snps), group=group)
        total = sum(parts)
    if total > UINT32_MAX:
        raise OverflowError(f"{total} SNPs over all ranks: a background bin could exceed the uint32 histogram")
    return total


def peer_setup(handle, group=None):
    """Map every rank's background histogram into every other rank (CUDA IPC over NVLink) for
    handle.peer_reduce_finalize().  Collective; the handle must hold its shard and tdsfs_background must have
    run once (single-group mode).  Returns False, leaving the NCCL path in use, when the mapping is not possible."""
    import torch.distributed as dist
    import tdsfs_capi as T
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    try:
        blob = handle.peer_export(rank, world)
    except T.TdsfsError:
        blob = None
    blobs = [None] * world
    dist.all_gather_object(blobs, blob, group=group)
    ok = all(b is not None for b in blobs)
    if ok:
        try:
            handle.peer_import(blobs)
        except T.TdsfsError:
            ok = False
    flags = [None] * world
    dist.all_gather_object(flags, ok, group=group)  # also the host barrier: every rank has mapped before anyone signals
    if not all(flags):
        handle.peer_close()
        return False
    return True


def peer_teardown(handle, group=None):
    """Collective: unmap the peers' histograms before any rank frees or re-shapes its own."""
    import torch
    import torch.distributed as dist
    torch.cuda.synchronize()
    dist.barrier(group=group)
    handle.peer_close()
    dist.barrier(group=group)


def _reduce_split_groups(handle, plan, rank, device, group=None):
    """Per-chromosome backgrounds with split chromosomes: sum the histograms of the pieces of each split chromosome over
    the ranks that hold them and write the sum back into every piece's group."""
    import torch
    import torch.distributed as dist
    owners = {}
    for r, pieces in enumerate(plan):
        for i, p in enumerate(pieces):
            owners.setdefault(p.chrom, []).append((r, i))
    split = sorted(c for c, o in owners.items() if len(o) > 1)
    if not split:
        return 0
    hist = background_tensor(handle, device)
    ng = max(len(plan[rank]), 1)
    gstride = hist.numel() // ng
    buf = torch.zeros((len(split), gstride), dtype=hist.dtype, device=hist.device)
    mine = {c: i for c, o in owners.items() for (r, i) in o if r == rank}
    for j, c in enumerate(split):
        if c in mine and plan[rank]:
            buf[j] = hist[mine[c] * gstride:(mine[c] + 1) * gstride]
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    for j, c in enumerate(split):
        if c in mine and plan[rank]:
            hist[mine[c] * gstride:(mine[c] + 1) * gstride] = buf[j]
    if hist.is_cuda:  # torch's stream wrote the sums back; the library's stream builds the tables next
        torch.cuda.current_stream(hist.device).synchronize()
    return len(split)


# ------------------------------------------------------------------------------------------------ results
def gather_results(local, chrom_base, group=None):
    """Concatenate per-rank result arrays in rank order (== the reference's sorted window order, because ranks own
    contiguous chromosome ranges).  local: dict name -> numpy array; chrom_base: global index of this rank's first chromosome."""
    import torch.distributed as dist
    local = dict(local)
    if "chrom" in local:
        local["chrom"] = local["chrom"] + np.int32(chrom_base)
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return local
    parts = [None] * dist.get_world_size(group)
    dist.all_gather_object(parts, local, group=group)
    return {k: np.concatenate([p[k] for p in parts]) for k in local}


def localize_results(res, pieces, pos, size, snp_mode):
    """A rank's result arrays (one entry per local candidate window) -> the entries the single-GPU scan holds for the same
    rows: local chromosome index -> global; the candidates a continuing fixed-bp piece shares with its predecessor (windows
    below its first SNP's window, empty here) dropped; the label of a continuing fixed-SNP piece's first window patched
    (previous SNP's position + 1, reference :1535)."""
    n = len(res["chrom"])
    keep = np.ones(n, dtype=bool)
    out = {k: v.copy() for k, v in res.items()}
    gl = np.array([p.chrom for p in pieces], dtype=np.int32) if pieces else np.zeros(0, np.int32)
    for i, p in enumerate(pieces):
        if p.first:
            continue
        sel = np.flatnonzero(res["chrom"] == i)
        if len(sel) == 0:
            continue
        if snp_mode:
            out["start"][sel[0]] = int(pos[p.lo - 1]) + 1
        else:
            k_prev = max(int(pos[p.lo - 1]) - 1, 0) // size      # last window of the predecessor piece
            keep[sel[:k_prev + 1]] = False
    if n:
        out["chrom"] = gl[res["chrom"]]
    return {k: v[keep] for k, v in out.items()}


def sharded_scan(handle, pieces, pos, size, bg_mode, device, *, snp_mode=False, bg_chrom=None, plan=None, rank=0, group=None,
                 peer=False):
    """plan -> background -> (exchange) -> finalize -> scan -> gather, for a handle that already holds this rank's pieces
    (loaded in order as its chromosomes).  pieces: this rank's entry of make_shard_plan; pos: positions of ALL SNPs; plan:
    the whole shard plan (needed for per-chromosome backgrounds with split chromosomes).  bg_chrom: GLOBAL chromosome
    index for BG_CHROM.  peer=True: the genome-wide / single-chromosome sum is the library's own peer-memory kernel (after
    peer_setup) instead of NCCL.  Returns the gathered result arrays (identical on every rank)."""
    n_local = sum(p.hi - p.lo for p in pieces)
    check_total_snps(n_local, group)
    if n_local:
        handle.plan(size, snp_mode=snp_mode)  # window boundaries on a side stream; arms the fused count kernel
    if bg_mode == BG_CHROM:
        local = [i for i, p in enumerate(pieces) if p.chrom == bg_chrom]
        handle.background(BG_CHROM, local[0] if local else -1)   # ranks without a piece of it contribute zeros
    else:
        handle.background(bg_mode)
    if bg_mode in (BG_GENOME, BG_CHROM):
        if peer:
            handle.peer_reduce_finalize()  # exchange + ln tables in one launch per rank
        else:
            allreduce_background(background_tensor(handle, device), group)
    elif bg_mode == BG_PER_CHROM and plan is not None:
        _reduce_split_groups(handle, plan, rank, device, group)
    handle.finalize_background()
    res = handle.scan(size, snp_mode=snp_mode)
    if hasattr(handle, "check"):
        handle.check()  # a late or missing peer must not pass as a result
    return gather_results(localize_results(res, pieces, pos, size, snp_mode), 0, group)



def sharded_diversity(handle, pieces, pos, size, device, *, snp_mode=False, group=None):
    """Per-window Hudson FST, pi and dxy of a sharded panel: the diversity counterpart of sharded_scan, for a handle that
    already holds this rank's pieces.  The sums of a window depend on its own rows only, so no collective is needed beyond
    the gather, and the gathered arrays equal a single-handle run bit for bit.  `device` is unused (the handle knows its
    GPU); it keeps sharded_scan's calling convention.  Returns the gathered arrays (identical on every rank)."""
    res = handle.diversity(size, snp_mode=snp_mode)
    return gather_results(localize_results(res, pieces, pos, size, snp_mode), 0, group)


def sharded_neutrality(handle, pieces, pos, size, device, *, snp_mode=False, group=None):
    """Per-window Watterson's theta and Tajima's D of a sharded panel: the neutrality counterpart of sharded_diversity,
    with the same calling convention.  Every result of a window depends on its own rows only (n is the window's largest
    called-allele count), so the gathered arrays equal a single-handle run bit for bit.  Returns the gathered arrays
    (identical on every rank)."""
    res = handle.neutrality(size, snp_mode=snp_mode)
    return gather_results(localize_results(res, pieces, pos, size, snp_mode), 0, group)


def sharded_wcfst(handle, pieces, pos, size, device, *, snp_mode=False, group=None):
    """Per-window Weir and Cockerham FST of a sharded panel (genotype entry): the counterpart of sharded_diversity, with
    the same calling convention.  Every result of a window depends on its own rows only, so the gathered arrays equal a
    single-handle run bit for bit.  Returns the gathered arrays (identical on every rank)."""
    res = handle.wcfst(size, snp_mode=snp_mode)
    return gather_results(localize_results(res, pieces, pos, size, snp_mode), 0, group)


def sharded_ld_windows(handle, pieces, pos, size, device, *, snp_mode=False, group=None):
    """Per-window ZnS and omega of a sharded panel (genotype entry): the counterpart of sharded_wcfst, with the same
    calling convention.  Every result of a window is a function of its own rows (exact integer sums), so the gathered
    arrays equal a single-handle run bit for bit.  Cost grows with the square of a window's rows.  Returns the gathered
    arrays (identical on every rank)."""
    res = handle.ld_windows(size, snp_mode=snp_mode)
    return gather_results(localize_results(res, pieces, pos, size, snp_mode), 0, group)
