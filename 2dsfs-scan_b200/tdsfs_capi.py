"""ctypes binding of libtdsfs.so (include/tdsfs.h) -- the thin host layer between the reference's Python API
and the hand-written CUDA kernels.  There is NO CPU fallback: if the library is missing or no CUDA device is
present every call raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libtdsfs.so")

BG_NONE, BG_PER_CHROM, BG_GENOME, BG_CHROM = 0, 1, 2, 3
F_T2D_NONE, F_T1D_P1_NONE, F_T1D_P2_NONE, F_EMPTY, F_SKIPPED = 1, 2, 4, 8, 16
ERR_ARG, ERR_CUDA, ERR_STATE, ERR_RANGE, ERR_RETRY = 1, 2, 3, 4, 5

EXPORTS = [
    "tdsfs_create", "tdsfs_destroy", "tdsfs_last_error", "tdsfs_set_stream", "tdsfs_set_sync", "tdsfs_set_panel",
    "tdsfs_load_counts", "tdsfs_load_genotypes", "tdsfs_background", "tdsfs_background_device", "tdsfs_get_background",
    "tdsfs_set_background", "tdsfs_finalize_background", "tdsfs_plan_bp", "tdsfs_plan_snp", "tdsfs_candidates_bp", "tdsfs_candidates_snp", "tdsfs_scan_bp",
    "tdsfs_scan_snp", "tdsfs_set_poisson_background", "tdsfs_scan_poisson_bp", "tdsfs_fetch_results", "tdsfs_check", "tdsfs_run_bp", "tdsfs_step_bp", "tdsfs_window_spectra", "tdsfs_likelihood",
    "tdsfs_poisson_score", "tdsfs_peer_export", "tdsfs_peer_import", "tdsfs_peer_allreduce_background", "tdsfs_peer_reduce_finalize", "tdsfs_peer_close",
    "tdsfs_synth_genotypes", "tdsfs_timings", "tdsfs_launch_count", "tdsfs_scan_info", "tdsfs_tail_stamps", "tdsfs_version",
    "tdsfs_diversity_bp", "tdsfs_diversity_snp", "tdsfs_fetch_diversity",
    "tdsfs_neutrality_bp", "tdsfs_neutrality_snp", "tdsfs_fetch_neutrality",
    "tdsfs_wcfst_bp", "tdsfs_wcfst_snp", "tdsfs_fetch_wcfst",
    "tdsfs_ld_prune",
    "tdsfs_ld_windows_bp", "tdsfs_ld_windows_snp", "tdsfs_fetch_ld_windows",
]


PEER_BLOB_BYTES = 192  # TDSFS_PEER_BLOB_BYTES
TIMING_NAMES = ("k1_count", "finalize", "k2_bounds", "k3_small", "k3_large", "background_call", "scan_call", "pass_total",
                "exchange", "diversity", "neutrality", "wcfst", "ld_pairs", "ld_resolve",
                "ld_windows")  # the slots of tdsfs_timings


class TdsfsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libtdsfs error {code}: {msg}")
        self.code = code


class Fixup(C.Structure):
    _fields_ = [("snp", C.c_int64), ("pop", C.c_int32), ("dref", C.c_int32), ("dalt", C.c_int32)]


FIXUP_DTYPE = np.dtype([("snp", "<i8"), ("pop", "<i4"), ("dref", "<i4"), ("dalt", "<i4")], align=True)


# Per-window result columns in the member order of tdsfs_result_t, tdsfs_diversity_t, tdsfs_neutrality_t, tdsfs_wcfst_t
# and tdsfs_ld_windows_t: each of those structs holds one host pointer per column.
RESULT_DTYPES = dict(chrom=np.int32, start=np.int64, end=np.int64, snp_count=np.int32, n2d=np.int32, n1d_p1=np.int32,
                     n1d_p2=np.int32, T2D=np.float64, T1D_p1=np.float64, T1D_p2=np.float64, flags=np.uint8)
DIVERSITY_DTYPES = dict(chrom=np.int32, start=np.int64, end=np.int64, snp_count=np.int32, flags=np.uint8, n_sites=np.int32,
                        pi_p1=np.float64, pi_p2=np.float64, dxy=np.float64, fst=np.float64)
NEUTRALITY_DTYPES = dict(chrom=np.int32, start=np.int64, end=np.int64, snp_count=np.int32, flags=np.uint8, n_seg_p1=np.int32,
                         n_seg_p2=np.int32, n_max_p1=np.int32, n_max_p2=np.int32, theta_pi_p1=np.float64,
                         theta_pi_p2=np.float64, theta_w_p1=np.float64, theta_w_p2=np.float64, tajima_d_p1=np.float64,
                         tajima_d_p2=np.float64)
WCFST_DTYPES = dict(chrom=np.int32, start=np.int64, end=np.int64, snp_count=np.int32, flags=np.uint8, n_sites=np.int32,
                    a=np.float64, b=np.float64, c=np.float64, fst=np.float64)
LD_WINDOWS_DTYPES = dict(chrom=np.int32, start=np.int64, end=np.int64, snp_count=np.int32, flags=np.uint8,
                         n_sites_p1=np.int32, n_sites_p2=np.int32, n_pairs_p1=np.int64, n_pairs_p2=np.int64,
                         zns_p1=np.float64, zns_p2=np.float64, omega_p1=np.float64, omega_p2=np.float64,
                         omega_pos_p1=np.int64, omega_pos_p2=np.int64)


class Result(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in RESULT_DTYPES]


class Diversity(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in DIVERSITY_DTYPES]


class Neutrality(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in NEUTRALITY_DTYPES]


class WcFst(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in WCFST_DTYPES]


class LdWindows(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in LD_WINDOWS_DTYPES]


_lib = None


def lib():
    """Load libtdsfs.so; raise loudly when it was not built (no silent fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TdsfsError(-1, f"{LIB_PATH} not found: build it with `python 2dsfs-scan_b200/build.py` "
                                 "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.tdsfs_last_error.restype = C.c_char_p
        L.tdsfs_launch_count.restype = C.c_int64
        L.tdsfs_launch_count.argtypes = [C.c_void_p]
        L.tdsfs_destroy.restype = None
        L.tdsfs_destroy.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def _ptr(a):
    """Host numpy array / device pointer holder / int / None -> void*."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if isinstance(a, int):
        return C.c_void_p(a)
    if hasattr(a, "data_ptr"):  # torch tensor (device or pinned host)
        return C.c_void_p(a.data_ptr())
    raise TypeError(type(a))


class Handle:
    """One GPU context (tdsfs_t)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        self._L = lib()
        self._keep = []  # keep host/device buffers adopted by the library alive
        self._check(self._L.tdsfs_create(C.c_int(device), C.byref(self._h)))
        self.n1 = self.n2 = 0
        self.C = 0
        self.S = 0

    def _check(self, rc):
        if rc != 0:
            raise TdsfsError(rc, self._L.tdsfs_last_error().decode())

    def close(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._L.tdsfs_destroy(h)
            self._h = None

    __del__ = close

    # ---- configuration
    def set_stream(self, stream_ptr):
        self._check(self._L.tdsfs_set_stream(self._h, C.c_void_p(stream_ptr or 0)))

    def set_sync(self, sync):
        self._check(self._L.tdsfs_set_sync(self._h, C.c_int(1 if sync else 0)))

    def set_panel(self, n1, n2, fold=True):
        self._check(self._L.tdsfs_set_panel(self._h, C.c_int32(n1), C.c_int32(n2), C.c_int32(1 if fold else 0)))
        self.n1, self.n2 = n1, n2

    # ---- data
    def load_counts(self, cnt, pos, chrom_off, flags=None):
        if isinstance(cnt, np.ndarray):
            cnt = np.ascontiguousarray(cnt, dtype=np.uint16)
            S = cnt.shape[0]
        else:
            S = int(cnt.shape[0])
        pos = np.ascontiguousarray(pos, dtype=np.int32) if isinstance(pos, np.ndarray) else pos
        off = np.ascontiguousarray(chrom_off, dtype=np.int64)
        if isinstance(flags, np.ndarray):
            flags = np.ascontiguousarray(flags, dtype=np.uint8)
        self._keep = [cnt, pos, off, flags]
        self.C = len(off) - 1
        self.S = int(S)
        self._check(self._L.tdsfs_load_counts(self._h, _ptr(cnt), C.c_int64(S), _ptr(pos), _ptr(off), C.c_int32(self.C), _ptr(flags)))

    def load_genotypes(self, G, S, words1, words2, ns1, ns2, pos, chrom_off, fixups=None, flags=None):
        if isinstance(G, np.ndarray):
            G = np.ascontiguousarray(G, dtype=np.uint32)
        pos = np.ascontiguousarray(pos, dtype=np.int32) if isinstance(pos, np.ndarray) else pos
        off = np.ascontiguousarray(chrom_off, dtype=np.int64)
        if isinstance(flags, np.ndarray):
            flags = np.ascontiguousarray(flags, dtype=np.uint8)
        nfix = 0
        if fixups is not None and len(fixups):
            fixups = np.ascontiguousarray(fixups, dtype=FIXUP_DTYPE)
            nfix = len(fixups)
        else:
            fixups = None
        self._keep = [G, pos, off, flags, fixups]
        self.C = len(off) - 1
        self.S = int(S)
        self._check(self._L.tdsfs_load_genotypes(self._h, _ptr(G), C.c_int64(S), C.c_int32(words1), C.c_int32(words2),
                                                 C.c_int32(ns1), C.c_int32(ns2), _ptr(pos), _ptr(off), C.c_int32(self.C),
                                                 _ptr(fixups), C.c_int64(nfix), _ptr(flags)))

    # ---- background
    def background(self, mode, bg_chrom=0, pos_lo=-1, pos_hi=-1):
        self._check(self._L.tdsfs_background(self._h, C.c_int32(mode), C.c_int32(bg_chrom), C.c_int64(pos_lo), C.c_int64(pos_hi)))

    def background_device(self):
        p, n, g = C.c_void_p(), C.c_int64(), C.c_int32()
        self._check(self._L.tdsfs_background_device(self._h, C.byref(p), C.byref(n), C.byref(g)))
        return p.value, n.value, g.value

    # ---- peer-memory exchange of the background (multi-GPU)
    def peer_export(self, rank, world):
        blob = C.create_string_buffer(PEER_BLOB_BYTES)
        self._check(self._L.tdsfs_peer_export(self._h, C.c_int32(rank), C.c_int32(world), blob))
        return blob.raw

    def peer_import(self, blobs):
        data = b"".join(blobs)
        self._check(self._L.tdsfs_peer_import(self._h, C.c_char_p(data)))

    def peer_allreduce_background(self):
        self._check(self._L.tdsfs_peer_allreduce_background(self._h))

    def peer_reduce_finalize(self):
        """All-reduce of the background and the ln tables in one launch (finalize_background afterwards is a no-op)."""
        self._check(self._L.tdsfs_peer_reduce_finalize(self._h))

    def peer_close(self):
        self._check(self._L.tdsfs_peer_close(self._h))

    def get_background(self, group=0):
        R1, R2 = 2 * self.n1 + 1, 2 * self.n2 + 1
        s2 = np.zeros(R1 * R2, dtype=np.uint64)
        s1a = np.zeros(R1, dtype=np.uint64)
        s1b = np.zeros(R2, dtype=np.uint64)
        self._check(self._L.tdsfs_get_background(self._h, C.c_int32(group), _ptr(s2), _ptr(s1a), _ptr(s1b)))
        return s2.reshape(R1, R2), s1a, s1b

    def set_background(self, b2d, b1a, b1b):
        R1, R2 = 2 * self.n1 + 1, 2 * self.n2 + 1
        b2d = np.ascontiguousarray(b2d, dtype=np.float64).reshape(-1)
        b1a = np.ascontiguousarray(b1a, dtype=np.float64)
        b1b = np.ascontiguousarray(b1b, dtype=np.float64)
        assert b2d.size == R1 * R2 and b1a.size == self.n1 + 1 and b1b.size == self.n2 + 1
        self._check(self._L.tdsfs_set_background(self._h, _ptr(b2d), _ptr(b1a), _ptr(b1b)))

    def set_poisson_background(self, q2d):
        """Normalised 2D background of the legacy Poisson score (dense (2n1+1) x (2n2+1), unfolded)."""
        R1, R2 = 2 * self.n1 + 1, 2 * self.n2 + 1
        q2d = np.ascontiguousarray(q2d, dtype=np.float64).reshape(-1)
        assert q2d.size == R1 * R2
        self._check(self._L.tdsfs_set_poisson_background(self._h, _ptr(q2d)))

    def scan_poisson(self, window_bp):
        """Poisson composite score of every fixed-bp window: dict of arrays, T2D = the score."""
        return self._into(self._alloc_result, self.candidates(window_bp, False), self._L.tdsfs_scan_poisson_bp,
                          C.c_int64(window_bp))

    def finalize_background(self):
        self._check(self._L.tdsfs_finalize_background(self._h))

    # ---- scans
    def plan(self, size, snp_mode=False):
        """Launch the window-boundary kernel ahead of the scan, on a side stream (overlaps background + all-reduce)."""
        f = self._L.tdsfs_plan_snp if snp_mode else self._L.tdsfs_plan_bp
        self._check(f(self._h, C.c_int64(size)))

    def candidates(self, size, snp_mode=False):
        n = C.c_int64()
        f = self._L.tdsfs_candidates_snp if snp_mode else self._L.tdsfs_candidates_bp
        self._check(f(self._h, C.c_int64(size), C.byref(n)))
        return n.value

    @staticmethod
    def _alloc(dtypes, struct, n):
        """Zeroed host arrays for n windows (at least one) and the result struct pointing at them."""
        arrs = {k: np.zeros(max(n, 1), dtype=dt) for k, dt in dtypes.items()}
        return arrs, struct(**{k: v.ctypes.data for k, v in arrs.items()})

    @staticmethod
    def _alloc_result(n):
        return Handle._alloc(RESULT_DTYPES, Result, n)

    @staticmethod
    def _alloc_diversity(n):
        return Handle._alloc(DIVERSITY_DTYPES, Diversity, n)

    @staticmethod
    def _alloc_neutrality(n):
        return Handle._alloc(NEUTRALITY_DTYPES, Neutrality, n)

    @staticmethod
    def _alloc_wcfst(n):
        return Handle._alloc(WCFST_DTYPES, WcFst, n)

    @staticmethod
    def _alloc_ld_windows(n):
        return Handle._alloc(LD_WINDOWS_DTYPES, LdWindows, n)

    def _into(self, alloc, cap, f, *args):
        """f(handle, *args, out, cap, &n) into the arrays alloc(cap) allocates: dict of their first n entries."""
        arrs, r = alloc(cap)
        n = C.c_int64()
        self._check(f(self._h, *args, C.byref(r), C.c_int64(cap), C.byref(n)))
        return {k: v[:n.value] for k, v in arrs.items()}

    def _run(self, entry, alloc, size, snp_mode, fetch):
        """Run tdsfs_<entry>_bp / _snp over the candidate windows of (size, mode): a dict of arrays, or the candidate count
        when fetch=False (the results stay on the device)."""
        f = getattr(self._L, f"tdsfs_{entry}_{'snp' if snp_mode else 'bp'}")
        if not fetch:
            n = C.c_int64()
            self._check(f(self._h, C.c_int64(size), None, C.c_int64(0), C.byref(n)))
            return n.value
        return self._into(alloc, self.candidates(size, snp_mode), f, C.c_int64(size))

    def scan(self, size, snp_mode=False, fetch=True):
        """Run K2 + K3/K4.  Returns dict of numpy arrays (one entry per candidate window) or the candidate count."""
        return self._run("scan", self._alloc_result, size, snp_mode, fetch)

    def diversity(self, size, snp_mode=False, fetch=True):
        """Per-window Hudson FST, pi and dxy over the candidate windows of (size, mode), in scan order (tdsfs_diversity_*).
        pi_p1 / pi_p2 / dxy are sums over the variant sites that entered (n_sites), not per-bp values; fst is NaN when
        dxy == 0.  Returns a dict of arrays (chrom / start / end / snp_count / flags as the scan's), or the candidate count
        when fetch=False (results stay on the device: fetch_diversity)."""
        return self._run("diversity", self._alloc_diversity, size, snp_mode, fetch)

    def fetch_diversity(self, cap):
        return self._into(self._alloc_diversity, cap, self._L.tdsfs_fetch_diversity)

    def neutrality(self, size, snp_mode=False, fetch=True):
        """Per-window, per-population Watterson's theta and Tajima's D over the candidate windows of (size, mode), in scan
        order (tdsfs_neutrality_*): n_seg_p* segregating sites, n_max_p* the largest called-allele count, theta_pi_p* /
        theta_w_p* absolute (not per-bp) estimators, tajima_d_p* at n = n_max_p* (NaN with fewer than 3 segregating sites).
        Returns a dict of arrays (chrom / start / end / snp_count / flags as the scan's), or the candidate count when
        fetch=False (results stay on the device: fetch_neutrality)."""
        return self._run("neutrality", self._alloc_neutrality, size, snp_mode, fetch)

    def fetch_neutrality(self, cap):
        return self._into(self._alloc_neutrality, cap, self._L.tdsfs_fetch_neutrality)

    def wcfst(self, size, snp_mode=False, fetch=True):
        """Per-window Weir and Cockerham (1984) FST over the candidate windows of (size, mode), in scan order
        (tdsfs_wcfst_*), from the genotype calls: a / b / c are the summed variance components (scikit-allel's
        weir_cockerham_fst summed over both alleles), n_sites the rows that entered a and b, fst = a / (a + b + c), NaN
        when that is 0.  Calls held as fix-ups count as missing.  Needs load_genotypes with at most 4000 samples per
        population.  Returns a dict of arrays (chrom / start / end / snp_count / flags as the scan's), or the candidate
        count when fetch=False (results stay on the device: fetch_wcfst)."""
        return self._run("wcfst", self._alloc_wcfst, size, snp_mode, fetch)

    def fetch_wcfst(self, cap):
        return self._into(self._alloc_wcfst, cap, self._L.tdsfs_fetch_wcfst)

    def ld_windows(self, size, snp_mode=False, fetch=True):
        """Per-window, per-population linkage disequilibrium over the candidate windows of (size, mode), in scan order
        (tdsfs_ld_windows_*), from the genotype calls: over the rows that pass the spectrum filter and each population's
        own samples, n_sites_p* the rows whose called dosages are not all equal, n_pairs_p* the row pairs with a defined
        r^2, zns_p* Kelly's ZnS (their mean r^2, NaN without pairs), omega_p* Kim and Nielsen's omega at its best split
        (NaN with fewer than 4 sites or no eligible split) and omega_pos_p* the position of the last site left of that
        split (-1 when omega is NaN).  r^2 enters as rint(r^2 2^32) in exact integer sums: results are bitwise
        reproducible.  Cost grows with the square of a window's rows.  Calls held as fix-ups count as missing.  Needs
        load_genotypes.  Returns a dict of arrays (chrom / start / end / snp_count / flags as the scan's), or the
        candidate count when fetch=False (results stay on the device: fetch_ld_windows)."""
        return self._run("ld_windows", self._alloc_ld_windows, size, snp_mode, fetch)

    def fetch_ld_windows(self, cap):
        return self._into(self._alloc_ld_windows, cap, self._L.tdsfs_fetch_ld_windows)

    def ld_prune(self, size, step, threshold):
        """LD pruning of the loaded genotype rows (tdsfs_ld_prune): scikit-allel's locate_unlinked(gn, size, step,
        threshold) per chromosome, r^2 over the samples of both populations called in both rows, exact integer sums with
        one rounded division.  Returns a bool array over the loaded rows, True = kept."""
        keep = np.zeros(max(self.S, 1), dtype=np.uint8)
        n = C.c_int64()
        self._check(self._L.tdsfs_ld_prune(self._h, C.c_int32(size), C.c_int32(step), C.c_double(threshold), _ptr(keep),
                                           C.byref(n)))
        out = keep[:self.S].astype(bool)
        assert int(out.sum()) == n.value
        return out

    def fetch_results(self, cap):
        return self._into(self._alloc_result, cap, self._L.tdsfs_fetch_results)

    def run_bp(self, bg_mode, W, fetch=True):
        if not fetch:
            n = C.c_int64()
            self._check(self._L.tdsfs_run_bp(self._h, C.c_int32(bg_mode), C.c_int64(W), None, C.c_int64(0), C.byref(n)))
            return n.value
        return self._into(self._alloc_result, self.candidates(W, False), self._L.tdsfs_run_bp, C.c_int32(bg_mode),
                          C.c_int64(W))

    def step_bp(self, bg_mode, W):
        """One whole asynchronous pass (CUDA graph after the first two calls); results stay on the device."""
        self._check(self._L.tdsfs_step_bp(self._h, C.c_int32(bg_mode), C.c_int64(W)))

    def window_spectra(self, window):
        R1, R2 = 2 * self.n1 + 1, 2 * self.n2 + 1
        s2 = np.zeros(R1 * R2, dtype=np.uint64)
        s1a = np.zeros(R1, dtype=np.uint64)
        s1b = np.zeros(R2, dtype=np.uint64)
        self._check(self._L.tdsfs_window_spectra(self._h, C.c_int64(window), _ptr(s2), _ptr(s1a), _ptr(s1b)))
        return s2.reshape(R1, R2), s1a, s1b

    def likelihood(self, x, b, B):
        """(value, is_none) of 2*(ll_fg - ll_bg) for interior count vector x against background values b."""
        x = np.ascontiguousarray(x, dtype=np.int64)
        b = np.ascontiguousarray(b, dtype=np.float64)
        T, flag = C.c_double(), C.c_int32()
        self._check(self._L.tdsfs_likelihood(self._h, _ptr(x), _ptr(b), C.c_int64(x.size), C.c_double(B), C.byref(T), C.byref(flag)))
        return T.value, bool(flag.value)

    def poisson_score(self, x, mu):
        x = np.ascontiguousarray(x, dtype=np.int64)
        mu = np.ascontiguousarray(mu, dtype=np.float64)
        out = C.c_double()
        self._check(self._L.tdsfs_poisson_score(self._h, _ptr(x), _ptr(mu), C.c_int64(x.size), C.byref(out)))
        return out.value

    # ---- synthetic + instrumentation
    def synth_genotypes(self, G_dev_ptr, S, snp0, words1, words2, ns1, ns2, seed, missing_rate=0.02, fst=0.05):
        self._check(self._L.tdsfs_synth_genotypes(self._h, C.c_void_p(G_dev_ptr), C.c_int64(S), C.c_int64(snp0), C.c_int32(words1),
                                                  C.c_int32(words2), C.c_int32(ns1), C.c_int32(ns2), C.c_uint64(seed),
                                                  C.c_double(missing_rate), C.c_double(fst)))

    def timings(self):
        ms = (C.c_float * len(TIMING_NAMES))()
        self._check(self._L.tdsfs_timings(self._h, ms, C.c_int32(len(ms))))
        return dict(zip(TIMING_NAMES, list(ms)))

    def diversity_ms(self):
        """CUDA-event time (ms) of the segment + finish kernels of the last diversity call (tdsfs_timings slot 9)."""
        return self.timings()["diversity"]

    def neutrality_ms(self):
        """CUDA-event time (ms) of the segment + finish kernels of the last neutrality call (tdsfs_timings slot 10)."""
        return self.timings()["neutrality"]

    def wcfst_ms(self):
        """CUDA-event time (ms) of the segment + finish kernels of the last wcfst call (tdsfs_timings slot 11)."""
        return self.timings()["wcfst"]

    def ld_prune_ms(self):
        """CUDA-event time (ms) of the pair and resolve kernels of the last ld_prune call (tdsfs_timings slots 12 + 13)."""
        t = self.timings()
        return t["ld_pairs"] + t["ld_resolve"]

    def ld_windows_ms(self):
        """CUDA-event time (ms) of the pair + finish kernels of the last ld_windows call (tdsfs_timings slot 14)."""
        return self.timings()["ld_windows"]

    def launch_count(self):
        return int(self._L.tdsfs_launch_count(self._h))

    def scan_info(self):
        """(fused, record_bytes) of the last scan: fused = the count kernel's window sums + the finish kernel scored it."""
        f, b = C.c_int32(), C.c_int32()
        self._check(self._L.tdsfs_scan_info(self._h, C.byref(f), C.byref(b)))
        return bool(f.value), int(b.value)

    def tail_stamps(self):
        """Diagnostics (TDSFS_TAIL_STAMPS=1): SM-clock stamps of CTA 0 at the phases of the count kernel's tail (8 x uint64)."""
        out = (C.c_uint64 * 8)()
        self._check(self._L.tdsfs_tail_stamps(self._h, out))
        return [int(x) for x in out]

    def check(self):
        """Synchronise and raise on deferred device-side errors (range, peer timeout, record overflow)."""
        self._check(self._L.tdsfs_check(self._h))
