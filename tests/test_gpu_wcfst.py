"""Per-window Weir and Cockerham (1984) FST (tdsfs_wcfst_*, wc_fst_scan): a numpy restatement of the definition in DESIGN.md
section 7, checked on the CPU against a literal restatement of scikit-allel's weir_cockerham_fst and
windowed_weir_cockerham_fst, then the GPU results against the restatement.

Definition, per row from the 2-bit codes alone (0 = 0/0, 1 = 0/1, 3 = 1/1, 2 = missing; calls held as fix-ups are missing):
n_i called diploids, x_i their alt alleles, h_i their heterozygotes; N = n1 + n2, X = x1 + x2, H = h1 + h2, D = x1 n2 - x2 n1;
a = [D^2 (N-1) - n1 n2 (X(2N-X) - N H)] / [4 n1^2 n2^2 (N-2)] and b = [n1 n2 (X(2N-X) - 2(N-1) H) - D^2] / [2 n1 n2 N (N-2)]
over the rows that pass the spectrum filter (snp_flags bit0) with n1 >= 1, n2 >= 1, N >= 3; c = H / N over the rows that pass
with N >= 1; exact integer numerators and denominators, one rounded division each; window sums in the order of the FST pass;
fst = a / ((a + b) + c), NaN when that is 0."""
import csv
import gzip
import os

import numpy as np
import pytest

from helpers import GOLDEN
from test_gpu_diversity import assert_bitwise, candidate_windows, random_codes, random_positions, window_sums

FLOATS = ("a", "b", "c", "fst")
INTS = ("chrom", "start", "end", "snp_count", "n_sites")


# ------------------------------------------------------------------------------------------- restatement (numpy)
def code_counts(c1, c2):
    """(n1, x1, h1, n2, x2, h2) per row of 2-bit codes [S, ns]."""
    out = []
    for c in (np.asarray(c1), np.asarray(c2)):
        out += [(c != 2).sum(1), (c == 1).sum(1) + 2 * (c == 3).sum(1), (c == 1).sum(1)]
    return [np.asarray(v, dtype=np.int64) for v in out]


def wc_terms(counts, passes=None):
    """(rows entering a and b, terms[S, 3] = a, b, c; +0.0 where a row adds no term).  Numerators and denominators are
    Python ints, converted to fp64 with round-to-nearest and divided once."""
    n1, x1, h1, n2, x2, h2 = counts
    N = n1 + n2
    ok = np.ones(len(n1), bool) if passes is None else np.asarray(passes, bool)
    ab = ok & (n1 >= 1) & (n2 >= 1) & (N >= 3)
    cm = ok & (N >= 1)
    n1, x1, h1, n2, x2, h2, N = (v.astype(object) for v in (n1, x1, h1, n2, x2, h2, N))
    X, H = x1 + x2, h1 + h2
    D = x1 * n2 - x2 * n1
    Q = X * (2 * N - X)
    a_num, a_den = D * D * (N - 1) - n1 * n2 * (Q - N * H), 4 * n1 * n1 * n2 * n2 * (N - 2)
    b_num, b_den = n1 * n2 * (Q - 2 * (N - 1) * H) - D * D, 2 * n1 * n2 * N * (N - 2)
    for v in (a_num[ab], a_den[ab], b_num[ab], b_den[ab]):
        assert all(abs(int(x)) < 2 ** 63 for x in v), "an int64 term would overflow"
    t = np.zeros((len(ab), 3))
    t[ab, 0] = a_num[ab].astype(np.float64) / a_den[ab].astype(np.float64)
    t[ab, 1] = b_num[ab].astype(np.float64) / b_den[ab].astype(np.float64)
    t[cm, 2] = H[cm].astype(np.float64) / N[cm].astype(np.float64)
    return ab, t


def restate(counts, pos, off, size, snp_mode=False, flags=None):
    """Arrays per candidate window, as tdsfs_wcfst_* returns them."""
    passes = None if flags is None else (np.asarray(flags) & 1) != 0
    counted = np.ones(len(counts[0]), np.int64) if flags is None else (np.asarray(flags, dtype=np.int64) >> 1) & 1
    ab, t = wc_terms(counts, passes)
    r = {k: [] for k in INTS + FLOATS + ("empty",)}
    for ch, lo, hi, st, en in candidate_windows(pos, off, size, snp_mode):
        s = window_sums(t, lo, hi)
        den = (s[0] + s[1]) + s[2]
        r["chrom"].append(ch); r["start"].append(st); r["end"].append(en); r["empty"].append(hi == lo)
        r["snp_count"].append(int(counted[lo:hi].sum())); r["n_sites"].append(int(ab[lo:hi].sum()))
        r["a"].append(s[0]); r["b"].append(s[1]); r["c"].append(s[2])
        r["fst"].append(np.nan if den == 0 else s[0] / den)
    return {k: np.array(v) for k, v in r.items()}


def gt_to_codes(g):
    """scikit-allel genotype array [S, ns, 2] without half calls -> 2-bit codes [S, ns]."""
    g = np.asarray(g)
    return np.where(g[:, :, 0] < 0, 2, np.array([0, 1, 3])[g.clip(0).sum(2)]).astype(np.uint8)


def codes_to_gt(c):
    """2-bit codes [S, ns] -> scikit-allel genotype array [S, ns, 2] (-1 = missing)."""
    lut = np.array([[0, 0], [0, 1], [-1, -1], [1, 1]])
    return lut[np.asarray(c)]


def skallel_wc_abc(g, subpops):
    """scikit-allel's _weir_cockerham_fst(g, subpops, max_allele=1) (allel/stats/fst.py), statement by statement:
    (a, b, c), each [S, 2 alleles], NaN where it divides by zero."""
    g = np.asarray(g)
    n_alleles, ploidy = 2, g.shape[2]
    r = len(subpops)
    with np.errstate(divide="ignore", invalid="ignore"):
        ac = np.dstack([np.stack([(g[:, sp] == al).sum(axis=(1, 2)) for al in range(n_alleles)], axis=1) for sp in subpops])
        an = np.sum(ac, axis=1)
        n = an / ploidy
        n_total = np.sum(n, axis=1)
        n_bar = np.mean(n, axis=1)
        n_C = (n_total - (np.sum(n ** 2, axis=1) / n_total)) / (r - 1)
        p = ac / an[:, np.newaxis, :]
        ac_total = np.sum(ac, axis=2)
        an_total = np.sum(an, axis=1)
        p_bar = ac_total / an_total[:, np.newaxis]
        n_bar = n_bar[:, np.newaxis]
        n_C = n_C[:, np.newaxis]
        n = n[:, np.newaxis, :]
        p_bar = p_bar[:, :, np.newaxis]
        s_squared = np.sum(n * ((p - p_bar) ** 2), axis=2) / (n_bar * (r - 1))
        p_bar = p_bar[:, :, 0]
        gs = g[:, np.concatenate(subpops)]
        called = (gs >= 0).all(axis=2)
        het = called & (gs[:, :, 0] != gs[:, :, 1])
        h_bar = np.column_stack([(het & (gs == al).any(axis=2)).sum(axis=1) / n_total for al in range(n_alleles)])
        a = ((n_bar / n_C) * (s_squared - ((1 / (n_bar - 1)) * ((p_bar * (1 - p_bar)) - ((r - 1) * s_squared / r)
                                                                 - (h_bar / 4)))))
        b = ((n_bar / (n_bar - 1)) * ((p_bar * (1 - p_bar)) - ((r - 1) * s_squared / r) - (((2 * n_bar) - 1) * h_bar / (4 * n_bar))))
        c = h_bar / 2
    return a, b, c


def skallel_window(a, b, c, rows):
    """windowed_weir_cockerham_fst's statistic on one window's rows: (sum a, sum b, sum c, fst) with np.nansum."""
    wa, wb, wc = np.nansum(a[rows]), np.nansum(b[rows]), np.nansum(c[rows])
    with np.errstate(divide="ignore", invalid="ignore"):
        return wa, wb, wc, wa / (wa + wb + wc)


def assert_skallel_close(exp, a, b, c, windows, passes, what="", eps=1e-12, strict_fst=True):
    """Restated windows vs scikit-allel's: equal n_sites (the rows where a is defined), the a, b and c sums within eps of
    the sums of their terms' magnitudes (a and b cancel).  fst within eps relative (strict_fst), else within the error
    those sums carry into a / (a + b + c)."""
    for w, (_, lo, hi, _, _) in enumerate(windows):
        rows = np.arange(lo, hi)[passes[lo:hi]]
        wa, wb, wc, f = skallel_window(a, b, c, rows)
        assert exp["n_sites"][w] == int(np.isfinite(a[rows, 0]).sum()), (what, w)
        mags = [np.nansum(np.abs(x[rows])) for x in (a, b, c)]
        for k, v, mag in zip("abc", (wa, wb, wc), mags):
            assert abs(exp[k][w] - v) <= eps * mag, (what, w, k, exp[k][w], v)
        assert np.isnan(exp["fst"][w]) == np.isnan(f), (what, w)
        if not np.isnan(f):
            tol = abs(f) if strict_fst else max(abs(f), (mags[0] + abs(f) * sum(mags)) / abs(wa + wb + wc))
            assert abs(exp["fst"][w] - f) <= eps * tol, (what, w, exp["fst"][w], f)


def rng_codes(rng, S, ns1, ns2):
    """Codes with heavy missingness, population-specific frequencies and rows that leave a, b (or c) undefined."""
    def codes(ns, f):
        a = (rng.random((S, ns)) < f[:, None]).astype(np.uint8) + (rng.random((S, ns)) < f[:, None]).astype(np.uint8)
        c = np.where(a == 2, 3, a).astype(np.uint8)
        c[rng.random((S, ns)) < rng.uniform(0.0, 0.6, S)[:, None]] = 2
        return c
    f = rng.uniform(0, 1, S)
    c1, c2 = codes(ns1, np.clip(f + rng.normal(0, 0.2, S), 0, 1)), codes(ns2, np.clip(f + rng.normal(0, 0.2, S), 0, 1))
    k = rng.choice(S, size=6 * (S // 50), replace=False).reshape(6, -1)
    c1[k[0]] = 2                         # population 1 uncalled: a, b NaN, c finite
    c2[k[1]] = 2                         # population 2 uncalled
    c1[k[2]] = 2; c2[k[2]] = 2           # nothing called: c NaN as well
    for r in k[3]:                       # n1 = n2 = 1: a, b NaN
        c1[r] = 2; c2[r] = 2; c1[r, 0] = rng.integers(0, 4) | 1; c2[r, 0] = rng.choice([0, 1, 3])
    c1[k[4]] = 1                         # all heterozygous
    c2[k[5], :] = 2; c2[k[5], :2] = 3    # n2 = 2
    return c1, c2


# ------------------------------------------------------------------------------------------- CPU: the restatement itself
def test_restatement_matches_scikit_allel():
    rng = np.random.default_rng(84)
    checked = 0
    for trial in range(10):
        S = int(rng.integers(300, 2500))
        ns1, ns2 = (int(v) for v in rng.integers(1, 40, size=2))
        c1, c2 = rng_codes(rng, S, ns1, ns2)
        pos = np.sort(rng.choice(np.arange(1, 40 * S), size=S, replace=False)).astype(np.int64)
        off = np.array([0, S // 3, S])
        flags = np.where(rng.random(S) < 0.1, 2, 3).astype(np.uint8)
        size = int(rng.choice([500, 5000, 20000]))
        exp = restate(code_counts(c1, c2), pos, off, size, flags=flags)
        a, b, c = skallel_wc_abc(np.concatenate([codes_to_gt(c1), codes_to_gt(c2)], axis=1),
                                 [np.arange(ns1), ns1 + np.arange(ns2)])
        wins = candidate_windows(pos, off, size, False)
        assert_skallel_close(exp, a, b, c, wins, (flags & 1) != 0, f"trial {trial}")
        checked += int(np.isfinite(exp["fst"]).sum())
    assert checked > 100


def test_restatement_known_cases():
    def one(c1, c2):
        c1, c2 = np.atleast_2d(c1).astype(np.uint8), np.atleast_2d(c2).astype(np.uint8)
        return restate(code_counts(c1, c2), np.arange(1, len(c1) + 1), [0, len(c1)], 10 ** 6)

    # a fixed difference without missing calls: a = 1, b = c = 0, fst = 1 exactly
    for ns1, ns2 in ((1, 2), (5, 3), (18, 14), (4000, 4000)):
        r = one(np.zeros(ns1), np.full(ns2, 3))
        assert (r["a"][0], r["b"][0], r["c"][0], r["fst"][0], r["n_sites"][0]) == (1.0, 0.0, 0.0, 1.0, 1), (ns1, ns2)
    r = one(np.zeros((7, 9)), np.full((7, 4), 3))
    assert (r["a"][0], r["b"][0], r["c"][0], r["fst"][0]) == (7.0, 0.0, 0.0, 1.0)
    # a monomorphic window: every term 0, fst undefined
    r = one(np.zeros((5, 6)), np.zeros((5, 6)))
    assert r["n_sites"][0] == 5 and r["a"][0] == 0 and r["b"][0] == 0 and r["c"][0] == 0 and np.isnan(r["fst"][0])
    # n1 = n2 = 1 and a population without calls add c only
    r = one([[1, 2, 2], [2, 2, 2]], [[3, 2], [1, 3]])
    assert r["n_sites"][0] == 0 and r["a"][0] == 0 and r["b"][0] == 0 and r["c"][0] == 0.5 + 1.0 / 2
    # equal frequencies in both populations: a < 0, so fst < 0
    r = one([[0, 3, 0, 3]] * 3, [[3, 0, 3, 0]] * 3)
    assert r["a"][0] < 0 and r["fst"][0] < 0


def test_save_csv_stats_wc_fst_column(tmp_path):
    import twoDSFS_class as K
    stats = {"c1 1-100": {"snp_count": 3, "T2D": 1.5, "T1D_pop1": None, "T1D_pop2": 0.25, "new_term_pop1": 1.0,
                          "new_term_pop2": 1.25, "T2D_diff": None},
             "c2 1-100": {"snp_count": 2, "T2D": 0.0, "T1D_pop1": 0.0, "T1D_pop2": 0.0, "new_term_pop1": 0.0,
                          "new_term_pop2": 0.0, "T2D_diff": 0.0},
             "c2 101-200": {"snp_count": 1, "T2D": 2.0, "T1D_pop1": 0.5, "T1D_pop2": 0.5, "new_term_pop1": 1.5,
                            "new_term_pop2": 1.5, "T2D_diff": 1.5}}
    wc = {"c1 1-100": {"snp_count": 3, "n_sites": 3, "a": 0.5, "b": 1.0, "c": 0.5, "FST": 0.25},
          "c2 1-100": {"snp_count": 2, "n_sites": 2, "a": 0.0, "b": 0.0, "c": 0.0, "FST": None}}
    path = tmp_path / "wc.csv"
    K.save_csv_stats(stats, str(path), fst=wc)
    rows = list(csv.reader(open(path, newline="")))
    assert rows[0][-1] == "FST" and len(rows[0]) == 11
    assert [r[-1] for r in rows[1:]] == ["0.25", "", ""]


def test_wc_fst_scan_rejects_a_data_dict():
    import twoDSFS_class as K
    from helpers import rows_to_dict
    inst = K.LikelihoodInference_jointSFS("x", "y")
    d = rows_to_dict([["c1", 10, [3, 1], [2, 2], "No annotation"]], ("uv", "bv"))
    for call in (lambda: inst.wc_fst_scan(d, 1000), lambda: inst.wc_fst_scan_bySNPs(d, 10)):
        with pytest.raises(TypeError, match="make_packed_panel"):
            call()


# ------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def T():
    import tdsfs_capi
    return tdsfs_capi


@pytest.fixture()
def h(T):
    hd = T.Handle(0)
    yield hd
    hd.close()


def assert_restated(res, exp, what=""):
    """GPU arrays per candidate window vs the restatement: equal labels and counts, bitwise equal sums and fst."""
    n = len(exp["start"])
    assert len(res["start"]) == n, (what, len(res["start"]), n)
    for k in INTS:
        assert np.array_equal(res[k], exp[k]), (what, k)
    assert np.array_equal((res["flags"] & 8) != 0, exp["empty"]), what
    for k in FLOATS:
        assert np.array_equal(res[k].view(np.uint64), exp[k].astype(np.float64).view(np.uint64)), (what, k)


def panel_codes(P):
    """2-bit codes [S, ns1], [S, ns2] of a PackedPanel (its fix-ups are not in them)."""
    from tdsfs_pack import from_b32, unpack_block
    rows = from_b32(P.G, P.n, P.W1 + P.W2)
    return unpack_block(rows[:, :P.W1], P.ns1), unpack_block(rows[:, P.W1:], P.ns2)


@pytest.mark.gpu
@pytest.mark.parametrize("ns1,ns2,S,C,L", [
    (200, 200, 40000, 4, 400000),    # 14 + 14 words (compile-time instantiation)
    (500, 500, 12000, 3, 120000),    # 32 + 32 words (compile-time instantiation)
    (100, 37, 20000, 5, 200000),     # 8 + 4 words: runtime word count, uneven split
    (2100, 2100, 4000, 2, 60000),    # 132 + 132 words: rows wider than 4096 samples
])
def test_genotype_panels_vs_restatement(T, h, ns1, ns2, S, C, L):
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(ns1 * 5 + ns2 + S)
    c1, c2 = random_codes(rng, S, ns1, ns2)
    c1[7], c2[7] = 2, 2
    c1[7, 3], c2[7, 1] = 1, 3  # n1 = n2 = 1
    pos, off = random_positions(rng, S, C, L)
    flags = np.where(rng.random(S) < 0.1, 2, 3).astype(np.uint8)
    flags[rng.random(S) < 0.05] &= 1
    G, w1, w2 = pack_codes(c1, c2)
    counts = code_counts(c1, c2)
    h.set_panel(ns1, ns2, True)
    h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off, flags=flags)
    defined = 0
    for size, snp in ((20000, False), (3000, False), (250, True), (1500, True)):
        a = h.wcfst(size, snp_mode=snp)
        assert_restated(a, restate(counts, pos, off, size, snp, flags), f"{size} {snp}")
        defined += int(np.isfinite(a["fst"]).sum())
    assert defined > 0


@pytest.mark.gpu
def test_ecb_subset_vcf_vs_restatement_and_scikit_allel():
    import twoDSFS_class as K
    vcf, pm = os.path.join(GOLDEN, "ecb_subset.vcf.gz"), os.path.join(GOLDEN, "ecb_subset.popmap.txt")
    inst = K.LikelihoodInference_jointSFS(vcf, pm)
    P = inst.make_packed_panel()
    # the VCF text: GT of every sample of uv (population 1) and bv (population 2), rows in the panel's order
    pop = dict(line.split()[:2] for line in open(pm) if len(line.split()) >= 2)
    recs = {}
    with gzip.open(vcf, "rt") as f:
        for line in f:
            if line.startswith("##"):
                continue
            cols = line.rstrip("\n").split("\t")
            if line.startswith("#"):
                names = cols[9:]
                continue
            gt = [s.split(":")[0] for s in cols[9:]]
            assert set(gt) <= {"0/0", "0/1", "1/1", "./."}
            row = [[int(x) if x != "." else -1 for x in g.split("/")] for g in gt]
            recs.setdefault(cols[0], []).append((int(cols[1]), row))
    sel = [[i for i, s in enumerate(names) if pop.get(s) == p] for p in (inst.pop1, inst.pop2)]
    g = []
    for c, chrom in enumerate(P.chroms):
        rows = sorted(recs[chrom], key=lambda r: r[0])
        assert [r[0] for r in rows] == P.pos[P.off[c]:P.off[c + 1]].tolist()
        g += [r[1] for r in rows]
    g = np.array(g)
    g = np.concatenate([g[:, sel[0]], g[:, sel[1]]], axis=1)
    ns1 = len(sel[0])
    a, b, c = skallel_wc_abc(g, [np.arange(ns1), ns1 + np.arange(len(sel[1]))])
    c1, c2 = panel_codes(P)
    counts = code_counts(c1, c2)
    for x, y in zip(counts, code_counts(gt_to_codes(g[:, :ns1]), gt_to_codes(g[:, ns1:]))):
        assert np.array_equal(x, y)
    passes = np.ones(P.n, bool)
    for size, snp in ((20000, False), (500000, False), (500, True)):
        got = inst.wc_fst_scan_bySNPs(P, size) if snp else inst.wc_fst_scan(P, size)
        eng = inst._eng()
        res = eng.h.fetch_wcfst(eng.h.candidates(size, snp))
        exp = restate(counts, P.pos, P.off, size, snp)
        assert_restated(res, exp, f"ecb {size}")
        # the literal restatement takes a dozen rounded steps per term: about 4e-12 relative each
        assert_skallel_close(exp, a, b, c, candidate_windows(P.pos, P.off, size, snp), passes, f"ecb {size}", 2e-11, False)
        live = ~exp["empty"]
        assert len(got) == int(live.sum()) and list(got) == list(inst.fst_scan(P, size) if not snp else inst.fst_scan_bySNPs(P, size))
        for v, k in zip(got.values(), np.flatnonzero(live)):
            assert list(v) == ["snp_count", "n_sites", "a", "b", "c", "FST"]
            assert v["a"] == exp["a"][k] and v["n_sites"] == exp["n_sites"][k]
            assert (v["FST"] is None) == bool(np.isnan(exp["fst"][k])) and (v["FST"] is None or v["FST"] == exp["fst"][k])
        assert any(v["FST"] is not None for v in got.values())


@pytest.mark.gpu
def test_fixups_count_as_missing_and_filters():
    import twoDSFS_class as K
    from tdsfs_engine import filter_flags
    vcf, pm = os.path.join(GOLDEN, "ingest_small.vcf.gz"), os.path.join(GOLDEN, "ingest_small.popmap.txt")
    inst = K.LikelihoodInference_jointSFS(vcf, pm, pop1_size=3, pop2_size=3)
    P = inst.make_packed_panel()
    assert P.fixups is not None and len(P.fixups) > 0
    c1, c2 = panel_codes(P)
    counts = code_counts(c1, c2)
    # the panel's allele counts are the codes' plus the fix-ups: the restatement leaves the fix-up calls out
    full = P.counts()
    for f in P.fixups:
        full[f["snp"], 2 * f["pop"]] -= f["dref"]
        full[f["snp"], 2 * f["pop"] + 1] -= f["dalt"]
    assert np.array_equal(full[:, 0] + full[:, 1], 2 * counts[0]) and np.array_equal(full[:, 1], counts[1])
    assert np.array_equal(full[:, 2] + full[:, 3], 2 * counts[3]) and np.array_equal(full[:, 3], counts[4])
    flags = filter_flags(P, None, None, None)
    for size, snp in ((30, False), (2, True)):
        got = inst.wc_fst_scan_bySNPs(P, size) if snp else inst.wc_fst_scan(P, size)
        eng = inst._eng()
        res = eng.h.fetch_wcfst(eng.h.candidates(size, snp))
        assert_restated(res, restate(counts, P.pos, P.off, size, snp, flags), f"ingest_small {size}")
        assert len(got) == int(((res["flags"] & 8) == 0).sum())
    # constructor filters: variant type on this panel, a position range on the ECB subset
    for vcf_, pm_, kw, ctor, size in (
            (vcf, pm, dict(pop1_size=3, pop2_size=3), dict(variant_type="missense_variant"), 30),
            (vcf, pm, dict(pop1_size=3, pop2_size=3), dict(start_position=8, end_position=60), 30),
            (os.path.join(GOLDEN, "ecb_subset.vcf.gz"), os.path.join(GOLDEN, "ecb_subset.popmap.txt"), {},
             dict(start_position=2_000_000, end_position=9_000_000), 100000)):
        inst = K.LikelihoodInference_jointSFS(vcf_, pm_, **kw, **ctor)
        P = inst.make_packed_panel()
        got = inst.wc_fst_scan(P, size)
        eng = inst._eng()
        res = eng.h.fetch_wcfst(eng.h.candidates(size))
        flags = filter_flags(P, ctor.get("start_position"), ctor.get("end_position"), ctor.get("variant_type"))
        counts = code_counts(*panel_codes(P))
        exp = restate(counts, P.pos, P.off, size, False, flags)
        assert_restated(res, exp, str(ctor))
        whole = restate(counts, P.pos, P.off, size, False)
        assert exp["c"].sum() < whole["c"].sum(), ctor
        assert len(got) == int((~exp["empty"]).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("size,snp", [(20000, False), (700, True)])
def test_shards_equal_whole_bitwise(T, size, snp):
    import tdsfs_dist as D
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(79)
    S, ns1, ns2 = 60000, 200, 200
    c1, c2 = random_codes(rng, S, ns1, ns2)
    pos, off = random_positions(rng, S, 2, 600000)
    plan = D.make_shard_plan(pos, off, 3, W=None if snp else size, N=size if snp else None, tol=0.0)
    assert any(not p.first for pieces in plan for p in pieces), "the plan must split a chromosome"
    h = T.Handle(0)
    try:
        h.set_panel(ns1, ns2, True)
        G, w1, w2 = pack_codes(c1, c2)
        h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
        whole = h.wcfst(size, snp_mode=snp)
        assert_restated(whole, restate(code_counts(c1, c2), pos, off, size, snp), "whole")
        parts, gathered = [], []
        for pieces in plan:
            a, b = pieces[0].lo, pieces[-1].hi
            Gr, _, _ = pack_codes(c1[a:b], c2[a:b])
            h.load_genotypes(Gr, b - a, w1, w2, ns1, ns2, pos[a:b], D.local_offsets(pieces))
            parts.append(D.localize_results(h.wcfst(size, snp_mode=snp), pieces, pos, size, snp))
            gathered.append(D.sharded_wcfst(h, pieces, pos, size, None, snp_mode=snp))
        for got in (parts, gathered):
            cat = {k: np.concatenate([p[k] for p in got]) for k in whole}
            assert_bitwise(cat, whole, "shards")
    finally:
        h.close()


@pytest.mark.gpu
def test_wcfst_does_not_disturb_the_scan_or_the_other_passes(T):
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(8)
    S, ns1, ns2, W = 30000, 200, 200, 20000
    c1, c2 = random_codes(rng, S, ns1, ns2)
    pos, off = random_positions(rng, S, 3, 300000)
    G, w1, w2 = pack_codes(c1, c2)

    def run(with_wc):
        h = T.Handle(0)
        try:
            h.set_panel(ns1, ns2, True)
            h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
            if with_wc:
                h.wcfst(5000, fetch=False)
            h.plan(W)
            if with_wc:
                h.wcfst(W, fetch=False)
            h.background(T.BG_GENOME)
            h.diversity(7000, fetch=False)
            h.neutrality(900, snp_mode=True, fetch=False)
            if with_wc:
                h.wcfst(900, snp_mode=True, fetch=False)
            h.finalize_background()
            res = h.scan(W)
            fused = h.scan_info()[0]
            div = h.fetch_diversity(h.candidates(7000))
            neut = h.fetch_neutrality(h.candidates(900, True))
            steps, others = [], []
            h.set_sync(False)
            for _ in range(3):
                h.step_bp(T.BG_GENOME, W)
                if with_wc:
                    h.wcfst(3000, snp_mode=True, fetch=False)
                h.diversity(W, fetch=False)
                h.neutrality(W, fetch=False)
                if with_wc:
                    h.wcfst(W, fetch=False)
                h.check()
                steps.append(h.fetch_results(h.candidates(W)))
                others += [h.fetch_diversity(h.candidates(W)), h.fetch_neutrality(h.candidates(W))]
            h.set_sync(True)
            return res, fused, [div, neut] + steps + others
        finally:
            h.close()

    a, fa, xa = run(True)
    b, fb, xb = run(False)
    assert fa and fb, "the planned scan must stay on the fused path"
    assert_bitwise(a, b, "scan")
    for x, y in zip(xa, xb):
        assert_bitwise(x, y, "step / diversity / neutrality")


@pytest.mark.gpu
def test_error_conventions(T, h):
    import ctypes as C
    from tdsfs_pack import pack_codes
    with pytest.raises(T.TdsfsError) as e:
        h.wcfst(1000)
    assert e.value.code == T.ERR_STATE
    h.set_panel(5, 5, True)
    with pytest.raises(T.TdsfsError) as e:
        h.fetch_wcfst(10)
    assert e.value.code == T.ERR_STATE
    # the counts entry has no heterozygote counts
    cnt = np.array([[4, 6, 5, 5]] * 100, dtype=np.uint16)
    pos = np.arange(1, 101, dtype=np.int32) * 50
    h.load_counts(cnt, pos, [0, 100])
    with pytest.raises(T.TdsfsError) as e:
        h.wcfst(1000)
    assert e.value.code == T.ERR_STATE and "genotype" in str(e.value)
    with pytest.raises(T.TdsfsError) as e:
        h.fetch_wcfst(100)
    assert e.value.code == T.ERR_STATE
    # more than 4000 samples in a population
    rng = np.random.default_rng(2)
    for ns1, ns2, ok in ((4001, 20, False), (20, 4001, False), (4000, 4000, True)):
        c1, c2 = random_codes(rng, 64, ns1, ns2)
        G, w1, w2 = pack_codes(c1, c2)
        h.load_genotypes(G, 64, w1, w2, ns1, ns2, np.arange(1, 65, dtype=np.int32) * 10, [0, 64])
        if ok:
            assert_restated(h.wcfst(300), restate(code_counts(c1, c2), np.arange(1, 65) * 10, [0, 64], 300), "4000 + 4000")
            continue
        with pytest.raises(T.TdsfsError) as e:
            h.wcfst(300)
        assert e.value.code == T.ERR_ARG and "4000" in str(e.value)
    c1, c2 = random_codes(rng, 100, 30, 30)
    G, w1, w2 = pack_codes(c1, c2)
    h.load_genotypes(G, 100, w1, w2, 30, 30, pos, [0, 100])
    for size in (0, -3):
        with pytest.raises(T.TdsfsError) as e:
            h.wcfst(size)
        assert e.value.code == T.ERR_ARG
    n = h.candidates(1000)
    arrs, r = h._alloc_wcfst(n)
    nw = C.c_int64()
    assert h._L.tdsfs_wcfst_bp(h._h, C.c_int64(1000), C.byref(r), C.c_int64(n - 1), C.byref(nw)) == T.ERR_ARG
    assert h._L.tdsfs_wcfst_bp(h._h, C.c_int64(1000), C.byref(r), C.c_int64(n), C.byref(nw)) == 0 and nw.value == n
    assert h.wcfst(1000, fetch=False) == n
    with pytest.raises(T.TdsfsError) as e:
        h.fetch_wcfst(n - 1)
    assert e.value.code == T.ERR_ARG
    # the other passes have their own results
    for fetch in (h.fetch_diversity, h.fetch_neutrality):
        with pytest.raises(T.TdsfsError) as e:
            fetch(n)
        assert e.value.code == T.ERR_STATE


@pytest.mark.gpu
def test_async_enqueue_then_fetch_equals_sync(T, h):
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(12)
    S, ns1, ns2 = 40000, 500, 500
    c1, c2 = random_codes(rng, S, ns1, ns2)
    pos, off = random_positions(rng, S, 3, 400000)
    G, w1, w2 = pack_codes(c1, c2)
    h.set_panel(ns1, ns2, True)
    h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
    want = {(size, snp): h.wcfst(size, snp_mode=snp) for size, snp in ((20000, False), (800, True))}
    h.set_sync(False)
    for (size, snp), exp in want.items():
        assert h.wcfst(size, snp_mode=snp, fetch=False) == len(exp["start"])
        assert_bitwise(h.fetch_wcfst(h.candidates(size, snp)), exp, f"async {size} {snp}")
    h.set_sync(True)
    assert h.wcfst_ms() > 0
