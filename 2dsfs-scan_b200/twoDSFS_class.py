"""Drop-in replacement for scripts/src/twoDSFS_class.py of uricchio/2DSFS-scan, backed by CUDA kernels for B200.

Same class name, constructor, method names, parameter order, defaults and return shapes as the reference
(class LikelihoodInference_jointSFS, reference lines 20-1736).  Every spectrum, window assignment and likelihood is
computed on the GPU through libtdsfs.so (C ABI, include/tdsfs.h); this file only adapts dicts to arrays and back and
reproduces the reference's observable quirks (SURVEY.md section 9): None for empty spectra, +inf for a populated
bin with zero background, the stale-carry of derived terms in combined_scan, the clobbered loop variable of T2D_scan,
the mis-indented sims_process_window, and the exceptions the unguarded scanners raise.  There is no CPU fallback:
without the built library or a CUDA device, calls raise.
"""
from __future__ import annotations

import csv
import glob
import gzip
import os

import numpy as np

import tdsfs_capi as T
from tdsfs_pack import PackedPanel, pack_vcf
from tdsfs_engine import (Engine, SnpTable, dense2d_to_dict, dict_to_dense2d, dict_to_folded1d, filter_flags, stat_lists,
                          window_keys)

_UNSET = object()


def _device():
    return int(os.environ.get("TDSFS_DEVICE", os.environ.get("LOCAL_RANK", "0")))


def parse_vcf_to_dict(vcf_filename, popinfo_filename):
    """Host-side ingest with the reference's exact gates (make_data_dict_vcf, reference :36-138): FILTER in {PASS, .},
    single-base A/C/G/T REF and ALT, annotation = 2nd '|' field of INFO, per-sample counting of the characters '0'/'1'
    at even offsets of the GT sub-field, and the positional population list (header samples found in the popmap, in
    order, zipped with the sample columns).  The text work runs in the C++ packer (tdsfs_pack.vcf_to_data_dict) when its
    library is built; the Python loop below is the same algorithm and the cross-check of the tests."""
    import tdsfs_pack
    if os.path.exists(tdsfs_pack._PACK_LIB) and not os.environ.get("TDSFS_PY_INGEST"):
        return tdsfs_pack.vcf_to_data_dict(vcf_filename, popinfo_filename)
    return _parse_vcf_to_dict_py(vcf_filename, popinfo_filename)


def _parse_vcf_to_dict_py(vcf_filename, popinfo_filename):
    popmap = {}
    with open(popinfo_filename, "r") as f:
        for line in f:
            cols = line.strip().split("\t")
            if len(cols) >= 2:
                popmap[cols[0]] = cols[1]
    data_dict = {}
    poplist = []
    acgt = ("A", "C", "G", "T")
    with gzip.open(vcf_filename, "rt") as f:
        for line in f:
            if line.startswith("##"):
                continue
            if line.startswith("#"):
                poplist.extend(popmap[s] for s in line.split()[9:] if s in popmap)
                continue
            cols = line.split("\t")
            info = cols[7].split("|")
            annotation = info[1] if len(info) >= 2 else "No annotation"
            if cols[6] != "PASS" and cols[6] != ".":
                continue
            ref, alt = cols[3].upper(), cols[4].upper()
            if ref not in acgt or alt not in acgt:
                continue
            gtindex = cols[8].split(":").index("GT")
            calls = {}
            for pop, sample in zip(poplist, cols[9:]):
                gt = sample.split(":")[gtindex][::2]
                r, a = calls.get(pop, (0, 0))
                calls[pop] = (r + gt.count("0"), a + gt.count("1"))
            data_dict["-".join(cols[:2])] = {"segregating": (ref, alt), "context": "-" + ref + "-", "calls": calls,
                                            "annotation": annotation}
    return data_dict


class LikelihoodInference_jointSFS:
    def __init__(self, vcf_filename, popinfo_filename, start_position=None, end_position=None,
                 pop1='uv', pop2='bv', pop1_size=18, pop2_size=14, variant_type=None, fold=True):
        self.vcf_filename = vcf_filename
        self.popinfo_filename = popinfo_filename
        self.pop1 = pop1
        self.pop2 = pop2
        self.pop1_size = pop1_size
        self.pop2_size = pop2_size
        self.start_position = start_position
        self.end_position = end_position
        self.variant_type = variant_type
        self.fold = fold
        self._engine = None
        self._tcache = None

    # ------------------------------------------------------------------ plumbing (not part of the reference API)
    def _eng(self):
        if self._engine is None:
            self._engine = Engine(_device())
        return self._engine

    def _table(self, data_dict, pop1=None, pop2=None):
        pop1 = self.pop1 if pop1 is None else pop1
        pop2 = self.pop2 if pop2 is None else pop2
        if isinstance(data_dict, PackedPanel):  # fast path: a VCF packed by make_packed_panel / tdsfs_pack.pack_vcf
            if (pop1, pop2) != tuple(data_dict.pops):
                raise TypeError(f"this PackedPanel holds populations {data_dict.pops}; {(pop1, pop2)} requested (use a data_dict)")
            return data_dict
        n = len(data_dict)
        tag = (id(data_dict), n, pop1, pop2, self._fingerprint(data_dict, n, pop1, pop2))
        if self._tcache is None or self._tcache[0] != tag:
            self._tcache = (tag, SnpTable.from_dict(data_dict, pop1, pop2))
        return self._tcache[1]

    @staticmethod
    def _fingerprint(data_dict, n, pop1, pop2, samples=512):
        """Content fingerprint of the array-form cache: first / last key and the (key, calls, annotation) of up to `samples`
        evenly spaced records.  The reference re-reads the dict on every call; the cache only skips the dict -> array
        conversion when the same dict object is scanned again.  An in-place edit of a record that is not sampled is NOT seen:
        call invalidate_cache() after mutating a data_dict between scans (or pass a new dict)."""
        if n == 0:
            return ()
        import itertools
        step = max(1, n // samples)
        out = [next(iter(data_dict)), next(reversed(data_dict))]
        for k, v in itertools.islice(data_dict.items(), 0, None, step):
            c = v.get("calls", {})
            out.append((k, c.get(pop1), c.get(pop2), v.get("annotation")))
        return hash(tuple(out))

    def invalidate_cache(self):
        """Forget the cached array form of the last data_dict (after editing a dict in place between scans)."""
        self._tcache = None

    def _int_filters(self):
        # calculate_2d_sfs coerces the position filters to int and stores them back (:168-171)
        if self.start_position is not None:
            self.start_position = int(self.start_position)
        if self.end_position is not None:
            self.end_position = int(self.end_position)

    def _flags(self, table):
        return filter_flags(table, self.start_position, self.end_position, self.variant_type)

    def _folded_bg(self, eng, group, which):
        _, s1a, s1b = eng.h.get_background(group)
        raw = s1a if which == 1 else s1b
        return self.fold_1d_sfs({i: int(v) for i, v in enumerate(raw.tolist())})

    # ------------------------------------------------------------------ ingest
    def make_data_dict_vcf(self, vcf_filename, popinfo_filename):
        return parse_vcf_to_dict(vcf_filename, popinfo_filename)

    def make_packed_panel(self, vcf_filename=None, popinfo_filename=None, nthreads=0):
        """Fast ingest (not in the reference): the same VCF + popmap rules as make_data_dict_vcf, packed by the C++ host
        packer into the 2-bit genotype matrix the GPU consumes.  The result can be passed to combined_scan, scan_chooseChr,
        scan_precomputed_BG, scan_*_bySNPs and calculate_2d_sfs wherever they take a data_dict."""
        return pack_vcf(vcf_filename or self.vcf_filename, popinfo_filename or self.popinfo_filename, self.pop1, self.pop2, nthreads)

    # ------------------------------------------------------------------ spectra
    def calculate_2d_sfs(self, data_dict):
        """reference :140-232.  Dense dict (i, j) -> count of the folded joint spectrum."""
        self.data_dict = data_dict
        self._int_filters()
        table = self._table(data_dict)
        h2, _, _ = self._eng().spectra(table, self.pop1_size, self.pop2_size, self.fold, self._flags(table))
        return dense2d_to_dict(h2.astype(np.int64))

    def normalize_2d_sfs(self, sfs):
        self.sfs = sfs
        counts = list(self.sfs.values())
        total = sum(counts[1:-1])
        return {coords: values / total for coords, values in self.sfs.items()}

    def calculate_p(self, foreground_sfs, background_sfs):
        """Legacy Poisson composite score (reference :249-289), SURVEY.md section 8(f) row f4."""
        self.foreground_sfs = foreground_sfs
        self.background_sfs = background_sfs
        keys = list(foreground_sfs.keys())
        S_w = sum(foreground_sfs.values())
        x = np.array([int(foreground_sfs[k]) for k in keys], dtype=np.int64)
        mu = np.array([S_w * background_sfs.get(k, 0) for k in keys], dtype=np.float64)
        return self._eng().h.poisson_score(x, mu)

    def count_snps(self, window_data, variant_type):
        self.window_data = window_data
        self.variant_type = variant_type  # (the reference overwrites the instance filter here, :294)
        snp_count = 0
        for snp_data in window_data.values():
            if variant_type is None or snp_data.get("annotation") == variant_type:
                snp_count += 1
        return snp_count

    def calculate_p_window(self, data_dict, sfs_normalized, window_size, pop1, pop2, pop1_size, pop2_size, start_position,
                           end_position, variant_type):
        """Broken in the reference (:304-393): the first window flush calls calculate_2d_sfs with nine arguments."""
        self.data_dict = data_dict
        self.sfs_normalized = sfs_normalized
        self.window_size = window_size
        self.pop1, self.pop2, self.pop1_size, self.pop2_size = pop1, pop2, pop1_size, pop2_size
        self.start_position, self.end_position, self.variant_type = start_position, end_position, variant_type
        if len(data_dict):
            raise TypeError("LikelihoodInference_jointSFS.calculate_2d_sfs() takes 2 positional arguments but 10 were given")
        return {}

    def calculate_1d_sfs(self, data_dict, pop, pop_size, start_position, end_position, variant_type):
        """reference :398-444.  Raw (unfolded) alt-count spectrum of one population."""
        self.data_dict = data_dict
        self.pop = pop
        self.pop_size = pop_size
        self.start_position = start_position
        self.end_position = end_position
        self.variant_type = variant_type
        if isinstance(data_dict, PackedPanel):
            if pop not in data_dict.pops:
                raise TypeError(f"this PackedPanel holds populations {data_dict.pops}")
            first = pop == data_dict.pops[0]
            n1, n2 = (pop_size, self.pop2_size) if first else (self.pop1_size, pop_size)
            flags = filter_flags(data_dict, start_position, end_position, variant_type)
            _, s1a, s1b = self._eng().spectra(data_dict, n1, n2, False, flags)
            return {i: int(v) for i, v in enumerate((s1a if first else s1b).tolist())}
        table = self._table(data_dict, pop, pop)
        flags = filter_flags(table, start_position, end_position, variant_type)
        _, s1, _ = self._eng().spectra(table, pop_size, pop_size, False, flags)
        return {i: int(v) for i, v in enumerate(s1.tolist())}

    def fold_1d_sfs(self, sfs_dict):
        num_chromosomes = max(sfs_dict.keys())
        folded = {}
        for freq, count in sfs_dict.items():
            m = min(freq, num_chromosomes - freq)
            folded[m] = folded[m] + count if m in folded else count
        return folded

    def normalize_1d_sfs(self, sfs):
        self.sfs = sfs
        counts = list(sfs.values())
        total = sum(counts[1:-1])
        return {freq: values / total for freq, values in sfs.items()}

    # ------------------------------------------------------------------ likelihoods
    def calculate_likelihood_1D(self, foreground_sfs, background_sfs):
        self.foreground_sfs = foreground_sfs
        self.background_sfs = background_sfs
        return self._eng().likelihood(foreground_sfs, background_sfs, guarded=True)

    def calculate_likelihood_2D(self, foreground_2d_sfs, background_2d_sfs):
        self.foreground_2d_sfs = foreground_2d_sfs
        self.background_2d_sfs = background_2d_sfs
        return self._eng().likelihood(foreground_2d_sfs, background_2d_sfs, guarded=True)

    def new_term(self, T1D, T2D):
        self.T1D = T1D
        self.T2D = T2D
        return T2D - T1D

    # ------------------------------------------------------------------ shared scan machinery
    def _scan(self, table, size, snp_mode, bg_mode=None, bg_chrom=0, precomputed=None, flags=_UNSET, cnt=None, n1=None, n2=None,
              fold=None):
        """Load + background + scan on the GPU.  Returns (keys, counts, [T2D, T1D_pop1, T1D_pop2] lists, live candidate ids, res)."""
        eng = self._eng()
        n1 = self.pop1_size if n1 is None else n1
        n2 = self.pop2_size if n2 is None else n2
        fl = self._flags(table) if flags is _UNSET else flags
        eng.load(table, n1, n2, self.fold if fold is None else fold, fl, cnt=cnt)
        # window boundaries ahead of the count kernel (side stream); with a PackedPanel (genotype entry) this also arms the
        # fused scan: the count kernel leaves every window's background-independent sums, one finish kernel scores them
        eng.h.plan(size, snp_mode=snp_mode)
        if precomputed is None:
            eng.background(bg_mode, bg_chrom)
            eng.h.finalize_background()
        else:
            eng.background(T.BG_NONE)
            eng.h.set_background(*precomputed)
        res = eng.scan(size, snp_mode)
        live = (res["flags"] & (T.F_EMPTY | T.F_SKIPPED)) == 0
        keys = window_keys(table, res, live)
        return keys, res["snp_count"][live].tolist(), stat_lists(res, live), np.flatnonzero(live), res

    @staticmethod
    def _nan_gate(values):
        """scipy returns NaN when the background is not a probability vector after normalisation (SURVEY 9.Q12)."""
        b = np.asarray(values, dtype=np.float64)
        B = b.sum()
        if B == 0:
            return False
        p = b / B
        return bool(abs(1.0 - p.sum()) > np.finfo(np.float64).eps * 10 or np.any(p < 0) or np.any(p > 1))

    def _precomputed(self, bg2, bg1a, bg1b):
        b2 = dict_to_dense2d(bg2, self.pop1_size, self.pop2_size)
        a = dict_to_folded1d(bg1a, self.pop1_size)
        b = dict_to_folded1d(bg1b, self.pop2_size)
        gates = (self._nan_gate(b2[1:-1]), self._nan_gate(a[1:-1]), self._nan_gate(b[1:-1]))
        return (b2, a, b), gates

    @staticmethod
    def _apply_gates(stats, gates):
        for s, g in zip(stats, gates):
            if g:
                for i, v in enumerate(s):
                    if v is not None:
                        s[i] = float("nan")

    def _unguarded(self, keys, counts, stats, with_diff=False, snp_count_fixed=None):
        """Result dict of the scanners without None guards (:1110, :1390, :1510): T2D - None raises TypeError."""
        results = {}
        for k, c, T2D, Ta, Tb in zip(keys, counts, *stats):
            if T2D is None or Ta is None or Tb is None:
                raise TypeError("unsupported operand type(s) for -: 'NoneType' and 'float'")
            rec = {"snp_count": c if snp_count_fixed is None else snp_count_fixed, "T2D": T2D, "T1D_pop1": Ta, "T1D_pop2": Tb,
                   "new_term_pop1": T2D - Ta, "new_term_pop2": T2D - Tb}
            if with_diff:
                rec["T2D_diff"] = T2D - (Ta + Tb) / 2
            results[k] = rec
        return results

    # ------------------------------------------------------------------ scanners
    def T1D_scan(self, data_dict, background_sfs, window_size, pop, pop_size):
        """reference :539-623."""
        self.data_dict = data_dict
        self.background_sfs = background_sfs
        self.window_size = window_size
        self.pop = pop
        self.pop_size = pop_size
        table = self._table(data_dict, pop, pop)
        if table.n == 0:
            return {}
        b1 = dict_to_folded1d(background_sfs, pop_size)
        gate = self._nan_gate(b1[1:-1])
        dummy2 = np.ones((2 * pop_size + 1) ** 2)
        keys, counts, stats, _, _ = self._scan(table, window_size, False, precomputed=(dummy2, b1, b1), n1=pop_size, n2=pop_size,
                                               fold=False)
        self._apply_gates(stats[1:2], (gate,))
        return {k: {"snp_count": c, "T1D": t} for k, c, t in zip(keys, counts, stats[1])}

    def T2D_scan(self, data_dict, background_2d_sfs, window_size):
        """reference :686-776, including its clobbered loop variable: the dead per-chromosome background loop (:740-742)
        rebinds `snp_key`, so the first SNP of every chromosome enters its window as the LAST-INSERTED key of data_dict."""
        self.data_dict = data_dict
        self.background_2d_sfs = background_2d_sfs
        self.window_size = window_size
        table = self._table(data_dict)
        if isinstance(table, PackedPanel):
            raise TypeError("T2D_scan needs a data_dict (its insertion-order quirk is not defined for a packed panel)")
        if table.n == 0:
            return {}
        self._int_filters()
        cnt = table.cnt.copy()
        flags = self._flags(table)
        flags = np.full(table.n, 3, dtype=np.uint8) if flags is None else flags.copy()
        lr = table.last_key_row
        sub_flag = flags[lr]
        firsts = table.off[:-1][np.diff(table.off) > 0]
        pos = table.pos
        for c, f in enumerate(firsts.tolist()):
            cnt[f] = table.cnt[lr]
            flags[f] = sub_flag
            # the substituted key can also be a genuine member of the same window: one dict entry, counted once
            if lr != f and table.off[c] <= lr < table.off[c + 1] and max(pos[lr] - 1, 0) // window_size == max(pos[f] - 1, 0) // window_size:
                flags[f] = 0
        b2 = dict_to_dense2d(background_2d_sfs, self.pop1_size, self.pop2_size)
        gate = self._nan_gate(b2[1:-1])
        ones1, ones2 = np.ones(self.pop1_size + 1), np.ones(self.pop2_size + 1)
        keys, counts, stats, _, _ = self._scan(table, window_size, False, precomputed=(b2, ones1, ones2), flags=flags, cnt=cnt)
        self._apply_gates(stats[0:1], (gate,))
        return {k: {"snp_count": c, "T2D": t} for k, c, t in zip(keys, counts, stats[0])}

    def combined_scan(self, data_dict, window_size):
        """reference :787-991: every chromosome its own background; stale-carry of the derived terms (:875/:930/:974)
        and the final-window block gated on the previous window's values (:952-989) are reproduced."""
        self.data_dict = data_dict
        self.window_size = window_size
        table = self._table(data_dict)
        if table.n == 0:
            raise UnboundLocalError("cannot access local variable 'T2D' where it is not associated with a value")
        self._int_filters()
        eng = self._eng()
        keys, counts, (T2, Ta, Tb), live_ids, res = self._scan(table, window_size, False, bg_mode=T.BG_PER_CHROM)
        results = {}
        nt1 = nt2 = diff = _UNSET
        nw = len(keys)

        def emit(i, T2D, T1, T2_):
            if nt1 is _UNSET:
                raise UnboundLocalError("cannot access local variable 'new_term_pop1' where it is not associated with a value")
            results[keys[i]] = {"snp_count": counts[i], "T2D": T2D, "T1D_pop1": T1, "T1D_pop2": T2_, "new_term_pop1": nt1,
                                "new_term_pop2": nt2, "T2D_diff": diff}

        for i in range(nw - 1):
            if T2[i] and Ta[i] and Tb[i] is not None:  # truthiness: None or 0.0 keeps the previous window's terms
                nt1, nt2, diff = T2[i] - Ta[i], T2[i] - Tb[i], T2[i] - (Ta[i] + Tb[i]) / 2
            emit(i, T2[i], Ta[i], Tb[i])
        # ---- final window (:952-989)
        last = nw - 1
        if nw < 2:
            raise UnboundLocalError("cannot access local variable 'T1D_pop1' where it is not associated with a value")
        chrom_last = int(res["chrom"][live_ids[last]])

        def folded_fg(i, which):
            _, s1a, s1b = eng.h.window_spectra(int(live_ids[i]))
            raw = s1a if which == 1 else s1b
            return self.fold_1d_sfs({j: int(v) for j, v in enumerate(raw.tolist())})

        T2D = T2[last]
        f1_from = last if T2D is not None else last - 1  # folded_fg_sfs_pop1 is refreshed only when T2D is not None
        T1 = Ta[last - 1]                                  # stale T1D_pop1 gates the next block (:963)
        if T1 is not None:
            T1 = Ta[last] if f1_from == last else eng.likelihood(folded_fg(f1_from, 1), self._folded_bg(eng, chrom_last, 1))
            f2_from = last
        else:
            f2_from = last - 1
        T2_ = Tb[last - 1]                                 # stale T1D_pop2 gates the emission (:970)
        if T2_ is not None:
            T2_ = Tb[last] if f2_from == last else eng.likelihood(folded_fg(f2_from, 2), self._folded_bg(eng, chrom_last, 2))
            if T2D and T1 and T2_ is not None:
                nt1, nt2, diff = T2D - T1, T2D - T2_, T2D - (T1 + T2_) / 2
            emit(last, T2D, T1, T2_)
        return results

    def scan_chooseChr(self, data_dict, window_size, background_chromosome):
        """reference :993-1159: one named chromosome is the background of every window."""
        self.data_dict = data_dict
        self.window_size = window_size
        table = self._table(data_dict)
        if background_chromosome not in table.chroms:
            raise ValueError(f"Background chromosome {background_chromosome} not found in the data.")
        self._int_filters()
        keys, counts, stats, _, _ = self._scan(table, window_size, False, bg_mode=T.BG_CHROM,
                                               bg_chrom=table.chroms.index(background_chromosome))
        return self._unguarded(keys, counts, stats)

    def scan_precomputed_BG(self, data_dict, window_size, bg_2d_sfs, bg_1d_sfs_pop1, bg_1d_sfs_pop2):
        """reference :1161-1299: backgrounds supplied by the caller (counts or normalised floats)."""
        self.data_dict = data_dict
        self.window_size = window_size
        table = self._table(data_dict)
        if table.n == 0:
            return {}
        self._int_filters()
        pre, gates = self._precomputed(bg_2d_sfs, bg_1d_sfs_pop1, bg_1d_sfs_pop2)
        keys, counts, stats, _, _ = self._scan(table, window_size, False, precomputed=pre)
        self._apply_gates(stats, gates)
        return self._unguarded(keys, counts, stats)

    def scan_chooseChr_bySNPs(self, data_dict, snp_window_size, background_chromosome):
        """reference :1303-1420: fixed-SNP windows, one chromosome as (normalised) background."""
        self.data_dict = data_dict
        self.snp_window_size = snp_window_size
        table = self._table(data_dict)
        if background_chromosome not in table.chroms:
            raise ValueError(f"Background chromosome {background_chromosome} not found in the data.")
        self._int_filters()
        # normalised backgrounds (:1334-1336): ZeroDivisionError when the chromosome has no interior SNP, as the reference
        c = table.chroms.index(background_chromosome)
        if isinstance(table, PackedPanel):
            raise TypeError("scan_chooseChr_bySNPs needs a data_dict (use scan_chooseChr / scan_perChr_bySNPs with a packed panel)")
        sub = SnpTable()
        lo, hi = int(table.off[c]), int(table.off[c + 1])
        sub.chroms, sub.off, sub.pos, sub.cnt, sub.ann, sub.keys, sub.pops, sub.n, sub.last_key_row = (
            [background_chromosome], np.array([0, hi - lo], dtype=np.int64), table.pos[lo:hi], table.cnt[lo:hi], table.ann[lo:hi],
            table.keys[lo:hi], table.pops, hi - lo, -1)
        h2, s1a, s1b = self._eng().spectra(sub, self.pop1_size, self.pop2_size, self.fold, self._flags(sub))
        bg2 = self.normalize_2d_sfs(dense2d_to_dict(h2.astype(np.int64)))
        bg1a = self.normalize_1d_sfs(self.fold_1d_sfs({i: int(v) for i, v in enumerate(s1a.tolist())}))
        bg1b = self.normalize_1d_sfs(self.fold_1d_sfs({i: int(v) for i, v in enumerate(s1b.tolist())}))
        pre, gates = self._precomputed(bg2, bg1a, bg1b)
        keys, counts, stats, _, _ = self._scan(table, snp_window_size, True, precomputed=pre)
        self._apply_gates(stats, gates)
        return self._unguarded(keys, counts, stats, snp_count_fixed=snp_window_size)

    def scan_perChr_bySNPs(self, data_dict, snp_window_size):
        """reference :1422-1541: fixed-SNP windows, every chromosome its own background."""
        self.data_dict = data_dict
        self.num_snps = snp_window_size
        table = self._table(data_dict)
        if table.n == 0:
            return {}
        self._int_filters()
        keys, counts, stats, _, _ = self._scan(table, snp_window_size, True, bg_mode=T.BG_PER_CHROM)
        return self._unguarded(keys, counts, stats, with_diff=True, snp_count_fixed=snp_window_size)

    # ------------------------------------------------------------------ diversity, neutrality, WC FST (not in the reference)
    def _window_pass(self, data_dict, size, snp_mode, entry):
        """Keys and result columns (lists) of the non-empty windows of (size, mode) from the per-window pass `entry`
        (Handle.diversity, .neutrality or .wcfst) over data_dict."""
        table = self._table(data_dict)
        if table.n == 0:
            return [], {}
        self._int_filters()
        eng = self._eng()
        eng.load(table, self.pop1_size, self.pop2_size, self.fold, self._flags(table))
        res = getattr(eng.h, entry)(size, snp_mode=snp_mode)
        live = (res["flags"] & T.F_EMPTY) == 0
        return window_keys(table, res, live), {k: v[live].tolist() for k, v in res.items()}

    def _fst(self, data_dict, size, snp_mode):
        keys, res = self._window_pass(data_dict, size, snp_mode, "diversity")
        if not keys:
            return {}
        cols = [res[k] for k in ("snp_count", "n_sites", "pi_p1", "pi_p2", "dxy", "fst")]
        return {k: {"snp_count": c, "n_sites": n, "pi_pop1": a, "pi_pop2": b, "dxy": d, "FST": None if f != f else f}
                for k, c, n, a, b, d, f in zip(keys, *cols)}

    def fst_scan(self, data_dict, window_size):
        """Hudson FST, pi and dxy of every non-empty fixed-bp window, computed on the GPU from the same data as the scans:
        {"{chrom} {start}-{end}": {"snp_count", "n_sites", "pi_pop1", "pi_pop2", "dxy", "FST"}}, keyed like combined_scan.
        A SNP enters the sums iff it passes the constructor's start_position / end_position / variant_type filters and has at
        least two called alleles in both populations.  pi_pop1 / pi_pop2 / dxy are SUMS over those n_sites variant sites, not
        per-bp values: divide by the window's callable length for per-bp diversity.  FST = 1 - (pi_pop1 + pi_pop2) / (2 dxy)
        (Hudson, as a ratio of averages: Bhatia et al. 2013 eq. 10; pixy --fst_type hudson), None when dxy == 0.
        snp_count is count_snps, as in the scanners.  Not in the reference; pass the result to save_csv_stats(fst=...)."""
        self.data_dict = data_dict
        self.window_size = window_size
        return self._fst(data_dict, window_size, False)

    def fst_scan_bySNPs(self, data_dict, snp_window_size):
        """fst_scan over fixed-SNP windows (full chunks of snp_window_size SNPs per chromosome, labelled like
        scan_perChr_bySNPs).  The key set is a superset of scan_perChr_bySNPs': a chunk that scanner skips because its 2D
        spectrum is empty has dxy == 0 here and appears with FST None.  snp_count is count_snps of the chunk (the scanner
        reports snp_window_size instead)."""
        self.data_dict = data_dict
        self.snp_window_size = snp_window_size
        return self._fst(data_dict, snp_window_size, True)

    _TAJIMA_COLS = dict(snp_count="snp_count", S_pop1="n_seg_p1", S_pop2="n_seg_p2", n_max_pop1="n_max_p1",
                        n_max_pop2="n_max_p2", theta_pi_pop1="theta_pi_p1", theta_pi_pop2="theta_pi_p2",
                        theta_w_pop1="theta_w_p1", theta_w_pop2="theta_w_p2", TajimaD_pop1="tajima_d_p1",
                        TajimaD_pop2="tajima_d_p2")

    def _tajima(self, data_dict, size, snp_mode):
        keys, res = self._window_pass(data_dict, size, snp_mode, "neutrality")
        if not keys:
            return {}
        cols = [res[c] for c in self._TAJIMA_COLS.values()]
        return {k: {name: None if v != v else v for name, v in zip(self._TAJIMA_COLS, row)} for k, row in zip(keys, zip(*cols))}

    def tajima_scan(self, data_dict, window_size):
        """Watterson's theta and Tajima's D of each population in every non-empty fixed-bp window, computed on the GPU from
        the same data as the scans: {"{chrom} {start}-{end}": {"snp_count", "S_pop1", "S_pop2", "n_max_pop1", "n_max_pop2",
        "theta_pi_pop1", "theta_pi_pop2", "theta_w_pop1", "theta_w_pop2", "TajimaD_pop1", "TajimaD_pop2"}}, keyed like
        fst_scan.  Per population, over the SNPs that pass the constructor's filters: S the segregating sites, n_max the
        largest number of called alleles, theta_pi the summed pairwise differences, theta_w = S / a1(n_max); Tajima's D is
        scikit-allel's tajima_d of the window's SNPs at n = n_max.  theta values are absolute, not per bp.  None where
        undefined: theta_w when n_max < 2, TajimaD when S < 3 or n_max == 2.  Negative D: an excess of rare variants
        (sweep, expansion); positive D: an excess of intermediate ones (balancing selection, structure).  Not in the
        reference; pass the result to save_csv_stats(tajima=...)."""
        self.data_dict = data_dict
        self.window_size = window_size
        return self._tajima(data_dict, window_size, False)

    def tajima_scan_bySNPs(self, data_dict, snp_window_size):
        """tajima_scan over fixed-SNP windows, with the windows and keys of fst_scan_bySNPs."""
        self.data_dict = data_dict
        self.snp_window_size = snp_window_size
        return self._tajima(data_dict, snp_window_size, True)

    def _wc_fst(self, panel, size, snp_mode):
        if not isinstance(panel, PackedPanel):
            raise TypeError("Weir and Cockerham FST needs the genotype calls: pass the PackedPanel of make_packed_panel "
                            "(a data_dict holds allele counts only, without heterozygotes)")
        keys, res = self._window_pass(panel, size, snp_mode, "wcfst")
        if not keys:
            return {}
        cols = [res[k] for k in ("snp_count", "n_sites", "a", "b", "c", "fst")]
        return {k: {"snp_count": c, "n_sites": n, "a": a, "b": b, "c": cc, "FST": None if f != f else f}
                for k, c, n, a, b, cc, f in zip(keys, *cols)}

    def wc_fst_scan(self, panel, window_size):
        """Weir and Cockerham's (1984) FST of every non-empty fixed-bp window, computed on the GPU from the genotype calls
        of a make_packed_panel panel: {"{chrom} {start}-{end}": {"snp_count", "n_sites", "a", "b", "c", "FST"}}, keyed like
        fst_scan.  a, b and c are the window's sums of scikit-allel's per-SNP variance components (weir_cockerham_fst,
        summed over both alleles) over the SNPs that pass the constructor's filters, and FST = a / (a + b + c), None when
        that is 0: scikit-allel's windowed_weir_cockerham_fst, the estimator of pixy's default FST column.  n_sites counts
        the SNPs with a called diploid in both populations and at least three in all, the ones that enter a and b.  Calls
        the packer holds as fix-ups (half calls, haploid and multi-allelic calls) count as missing.  At most 4000 samples
        per population.  Not in the reference; pass the result to save_csv_stats(fst=...)."""
        self.window_size = window_size
        return self._wc_fst(panel, window_size, False)

    def wc_fst_scan_bySNPs(self, panel, snp_window_size):
        """wc_fst_scan over fixed-SNP windows, with the windows and keys of fst_scan_bySNPs."""
        self.snp_window_size = snp_window_size
        return self._wc_fst(panel, snp_window_size, True)

    # ------------------------------------------------------------------ LD pruning (not in the reference)
    def ld_prune(self, panel, size=100, step=20, threshold=0.1):
        """Drop the SNPs in linkage disequilibrium from a make_packed_panel panel, on the GPU: scikit-allel's
        locate_unlinked(gn, size, step, threshold) (defaults are its own), the windowed greedy r^2 rule of PLINK's
        --indep-pairwise.  Per chromosome, windows of `size` SNPs start every `step` SNPs; walking the SNPs in order, a SNP
        is dropped when its r^2 with an earlier kept SNP of a common window exceeds `threshold`.  r^2 is the squared
        correlation of the alt-allele dosages (0, 1, 2) over the samples of both populations called at both SNPs; calls the
        packer holds as fix-ups (half calls, haploid and multi-allelic calls) count as missing.  The constructor's
        start_position / end_position / variant_type filters are NOT applied: pruning covers every SNP of the panel, and
        the scans apply their filters to the pruned panel afterwards.  Returns the pruned PackedPanel (tdsfs_pack.subset_panel),
        which every scan and window pass accepts; its ld_prune attribute holds (size, step, threshold).  2 <= size <= 1024,
        step >= 1, threshold in [0, 1].  Not in the reference, which reads VCFs pruned beforehand with PLINK."""
        if not isinstance(panel, PackedPanel):
            raise TypeError("LD pruning needs the genotype calls: pass the PackedPanel of make_packed_panel "
                            "(a data_dict holds allele counts only, without genotypes)")
        import tdsfs_pack
        eng = self._eng()
        eng.load(panel, self.pop1_size, self.pop2_size, self.fold)
        keep = eng.h.ld_prune(int(size), int(step), float(threshold))
        return tdsfs_pack.subset_panel(panel, keep, (size, step, threshold))

    # ------------------------------------------------------------------ simulations
    def get_gens(self, main_dir):
        search_strings = set()
        for root, dirs, files in os.walk(main_dir):
            for file in files:
                parts = file.split('.')
                if len(parts) == 5:
                    search_strings.add(parts[1])
        return search_strings

    def sims_process_window(self, data_dict, window_size, bg_2d_sfs, bg_p1_sfs, bg_p2_sfs):
        """reference :1555-1687.  Its window logic is nested inside the chromosome-change branch (:1617-1654), so only
        the FIRST SNP of each chromosome ever enters a window (snp_count == 1); reproduced as is."""
        self.data_dict = data_dict
        self.window_size = window_size
        table = self._table(data_dict)
        if isinstance(table, PackedPanel):
            raise TypeError("sims_process_window needs a data_dict")
        if table.n == 0:
            return {}
        self._int_filters()
        firsts = table.off[:-1][np.diff(table.off) > 0]
        sub = SnpTable()
        sub.chroms, sub.pos, sub.cnt, sub.ann = table.chroms, table.pos[firsts], table.cnt[firsts], table.ann[firsts]
        sub.keys, sub.pops, sub.n, sub.last_key_row = [table.keys[i] for i in firsts.tolist()], table.pops, len(firsts), -1
        sub.off = np.concatenate([[0], np.cumsum((np.diff(table.off) > 0).astype(np.int64))]).astype(np.int64)
        pre, gates = self._precomputed(bg_2d_sfs, bg_p1_sfs, bg_p2_sfs)
        keys, counts, stats, live_ids, res = self._scan(sub, window_size, False, precomputed=pre)
        self._apply_gates(stats, gates)
        results = {}
        starts = res["start"][live_ids].tolist()
        for k, st, T2D, Ta, Tb in zip(keys, starts, *stats):
            if T2D is None or Ta is None or Tb is None:
                raise TypeError("unsupported operand type(s) for -: 'NoneType' and 'float'")
            results[k] = {"window_type": "background" if 0 <= st < 500000 else "foreground", "window_start": st,
                          "window_end": st + window_size, "snp_count": 1, "T2D": T2D, "T1D_p1": Ta, "T1D_p2": Tb,
                          "new_term_p1": T2D - Ta, "new_term_p2": T2D - Tb}
        return results

    def scan_sims(self, main_dir, window_size):
        """reference :1690-1736 (returns only the last replicate's dict, like the reference).  The reference hard-codes a
        popmap path on the author's machine; this uses it when it exists and the constructor's popinfo_filename otherwise."""
        self.main_dir = main_dir
        self.window_size = window_size
        hard = "/Users/marlonalejandrocalderonbalcazar/Desktop/ECB/simulations/results/popmap_sims_copy.txt"
        popinfo_filename = hard if os.path.exists(hard) else self.popinfo_filename
        generations = self.get_gens(main_dir)
        for generation in generations:
            target_vcfs = glob.glob(f"{main_dir}/iter*/*{generation}*.vcf.gz")
            concatenated_vcfs = glob.glob(f"{main_dir}/concatenated_vcfs/gen.{generation}.concatenated.vcf.gz")
            for vcf in concatenated_vcfs:
                data_dict = self.make_data_dict_vcf(vcf, popinfo_filename)
                bg_snps = {k: v for k, v in data_dict.items() if int(k.split('-')[1]) <= 500000}
                bg_2d_sfs = self.calculate_2d_sfs(bg_snps)
                bg_p1_sfs = self.fold_1d_sfs(self.calculate_1d_sfs(bg_snps, self.pop1, self.pop1_size, self.start_position,
                                                                  self.end_position, self.variant_type))
                bg_p2_sfs = self.fold_1d_sfs(self.calculate_1d_sfs(bg_snps, self.pop2, self.pop2_size, self.start_position,
                                                                  self.end_position, self.variant_type))
                for vcf_input in target_vcfs:
                    iteration_number = int(vcf_input.split('.')[2])  # noqa: F841 (computed and unused in the reference too)
                    data_dict_target = self.make_data_dict_vcf(vcf_input, popinfo_filename)
                    sims_stats = self.sims_process_window(data_dict_target, window_size, bg_2d_sfs, bg_p1_sfs, bg_p2_sfs)
        return sims_stats


# ---------------------------------------------------------------------- module-level helpers of the reference
chr_ids = {}


def load_chr_ids(chromosomes_txt):
    """chromosomes.txt (accession -> chromosome number); the reference loads it at import from a hard-coded path (:1788-1797)."""
    out = {}
    with open(chromosomes_txt) as f:
        next(f, None)
        for line in f:
            p = line.split()
            if len(p) >= 2:
                out[p[0]] = p[1]
    chr_ids.clear()
    chr_ids.update(out)
    return out


col_names = ['chromosome', 'window_start', 'window_end', 'snp_count', 'T2D', 'T1D_p1', 'T1D_p2', 'new_term_p1', 'new_term_p2', 'T2D_diff']


def save_csv_stats(stats_dict, output, fst=None, tajima=None):
    """reference :1884-1907: same columns, chromosome mapped through chr_ids, None written as ''.  fst (not in the
    reference): the dict of fst_scan / fst_scan_bySNPs or wc_fst_scan / wc_fst_scan_bySNPs over the same windows adds a
    trailing FST column, the layout of the ECB tables the reference's R post-processing writes; '' where FST is None or
    the window has no entry.  tajima (not in the reference): the dict of tajima_scan / tajima_scan_bySNPs adds TajimaD_p1,
    TajimaD_p2 after it, '' likewise."""
    with open(output, 'w', newline='') as csvfile:
        writer = csv.DictWriter(csvfile, fieldnames=col_names + (['FST'] if fst is not None else [])
                                + (['TajimaD_p1', 'TajimaD_p2'] if tajima is not None else []))
        writer.writeheader()
        for window_coords, result in stats_dict.items():
            chromosome = window_coords.split(' ')[0]
            window_start, window_end = window_coords.split(' ')[1].split('-')
            row = {'chromosome': chr_ids.get(chromosome, chromosome), 'window_start': window_start, 'window_end': window_end,
                   'snp_count': result["snp_count"], 'T2D': result["T2D"], 'T1D_p1': result["T1D_pop1"],
                   'T1D_p2': result["T1D_pop2"], 'new_term_p1': result["new_term_pop1"],
                   'new_term_p2': result["new_term_pop2"], 'T2D_diff': result["T2D_diff"]}
            if fst is not None:
                row['FST'] = fst.get(window_coords, {}).get("FST")
            if tajima is not None:
                t = tajima.get(window_coords, {})
                row['TajimaD_p1'], row['TajimaD_p2'] = t.get("TajimaD_pop1"), t.get("TajimaD_pop2")
            writer.writerow(row)


def plot_2d_sfs(*args, **kwargs):
    raise NotImplementedError("plotting (reference :1739-1786) is outside the B200 hot path; use the reference's matplotlib code "
                              "on the dicts returned by this class")


def plot_manhattan(*args, **kwargs):
    raise NotImplementedError("plotting (reference :1800-1878) is outside the B200 hot path; use save_csv_stats + ECBstats_plots.R")
