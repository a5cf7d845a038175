"""Per-window Watterson's theta and Tajima's D (tdsfs_neutrality_*, tajima_scan): a numpy restatement of the definition in
DESIGN.md section 7, checked on the CPU against a literal restatement of scikit-allel's tajima_d, then the GPU results
against the restatement.

Definition, per population i over the rows that pass the spectrum filters (snp_flags bit0), n_i = ref_i + alt_i:
S_i = #rows with ref_i > 0 and alt_i > 0; n_max_i = max n_i (0 without rows); theta_pi_i = sum over rows with n_i >= 2 of
2 ref_i alt_i / (n_i (n_i - 1)) in the summation order of the FST pass; theta_w_i = S_i / a1(n_max_i) (NaN when
n_max_i < 2); Tajima's D with Tajima's (1989) constants at n = n_max_i, NaN when S_i < 3 or the variance term is not > 0."""
import csv
import os

import numpy as np
import pytest

from helpers import GOLDEN, load_chr1_dict
from test_gpu_diversity import (assert_bitwise, candidate_windows, codes_to_counts, random_codes, random_positions,
                                window_sums)

FLOATS = ("theta_pi_p1", "theta_pi_p2", "theta_w_p1", "theta_w_p2", "tajima_d_p1", "tajima_d_p2")
INTS = ("chrom", "start", "end", "snp_count", "n_seg_p1", "n_seg_p2", "n_max_p1", "n_max_p2")


# ------------------------------------------------------------------------------------------- restatement (numpy)
def harmonic_tables(nmax):
    """a1[n] = sum_{k=1}^{n-1} 1/k and a2[n] = sum_{k=1}^{n-1} 1/k^2 for n in [0, nmax], summed in ascending k."""
    k = np.arange(1, max(nmax, 1), dtype=np.float64)
    return np.concatenate([[0.0, 0.0], np.cumsum(1.0 / k)]), np.concatenate([[0.0, 0.0], np.cumsum(1.0 / (k * k))])


def tajima_constants(n, a1, a2):
    """(e1, e2) of Tajima (1989) at sample size n."""
    b1 = (n + 1) / (3 * (n - 1))
    b2 = 2 * (n * n + n + 3) / (9 * n * (n - 1))
    c1 = b1 - 1 / a1
    c2 = b2 - (n + 2) / (a1 * n) + a2 / (a1 * a1)
    return c1 / a1, c2 / (a1 * a1 + a2)


def neutrality_stats(pi, S, n, a1t, a2t):
    """(theta_w, D) of one population of one window."""
    if n < 2:
        return np.nan, np.nan
    a1, a2 = a1t[n], a2t[n]
    tw = S / a1
    if S < 3:
        return tw, np.nan
    e1, e2 = tajima_constants(n, a1, a2)
    var = e1 * S + e2 * S * (S - 1)
    return tw, (pi - tw) / np.sqrt(var) if var > 0 else np.nan


def restate(cnt, pos, off, size, snp_mode=False, flags=None):
    """Arrays per candidate window, as tdsfs_neutrality_* returns them."""
    c = np.asarray(cnt, dtype=np.int64).reshape(-1, 4)
    passes = np.ones(len(c), bool) if flags is None else (np.asarray(flags) & 1) != 0
    counted = np.ones(len(c), np.int64) if flags is None else (np.asarray(flags, dtype=np.int64) >> 1) & 1
    terms, seg, nmx = np.zeros((len(c), 2)), [], []
    for i in range(2):
        r, a = c[:, 2 * i], c[:, 2 * i + 1]
        n = r + a
        e = passes & (n >= 2)
        terms[e, i] = (2 * r[e] * a[e]).astype(np.float64) / (n[e] * (n[e] - 1)).astype(np.float64)
        seg.append(passes & (r > 0) & (a > 0))
        nmx.append(np.where(passes, n, 0))
    a1t, a2t = harmonic_tables(int(max(nmx[0].max(initial=0), nmx[1].max(initial=0))))
    out = {k: [] for k in INTS + FLOATS + ("empty",)}
    for ch, lo, hi, st, en in candidate_windows(pos, off, size, snp_mode):
        s = window_sums(terms, lo, hi)
        out["chrom"].append(ch); out["start"].append(st); out["end"].append(en); out["empty"].append(hi == lo)
        out["snp_count"].append(int(counted[lo:hi].sum()))
        for i in range(2):
            S, n = int(seg[i][lo:hi].sum()), int(nmx[i][lo:hi].max(initial=0))
            tw, d = neutrality_stats(s[i], S, n, a1t, a2t)
            p = f"_p{i + 1}"
            out["n_seg" + p].append(S); out["n_max" + p].append(n); out["theta_pi" + p].append(s[i])
            out["theta_w" + p].append(tw); out["tajima_d" + p].append(d)
    return {k: np.array(v) for k, v in out.items()}


def skallel_tajima_d(ac, min_sites=3):
    """scikit-allel's tajima_d(ac) (allel/stats/diversity.py), statement by statement, for biallelic counts ac[S, 2]:
    (S, n, theta_w, D), theta_w = S / a1 as it computes it on the way."""
    ac = np.asarray(ac, dtype=np.int64)
    S = int(np.count_nonzero(np.sum(ac > 0, axis=1) > 1))      # ac.count_segregating()
    n = int(ac.sum(axis=1).max()) if len(ac) else 0             # ac.sum(axis=1).max()
    a1 = np.sum(1 / np.arange(1, n))
    with np.errstate(divide="ignore", invalid="ignore"):
        theta_hat_w_abs = S / a1
    if S < min_sites:
        return S, n, theta_hat_w_abs, np.nan
    an = np.sum(ac, axis=1)                                     # mean_pairwise_difference(ac, fill=0)
    n_pairs = an * (an - 1) / 2
    n_same = np.sum(ac * (ac - 1) / 2, axis=1)
    n_diff = n_pairs - n_same
    with np.errstate(divide="ignore", invalid="ignore"):
        mpd = np.where(n_pairs > 0, n_diff / n_pairs, 0.0)
    theta_hat_pi_abs = np.sum(mpd)
    d = theta_hat_pi_abs - theta_hat_w_abs
    a2 = np.sum(1 / (np.arange(1, n) ** 2))
    b1 = (n + 1) / (3 * (n - 1))
    b2 = 2 * (n ** 2 + n + 3) / (9 * n * (n - 1))
    c1 = b1 - (1 / a1)
    c2 = b2 - ((n + 2) / (a1 * n)) + (a2 / (a1 ** 2))
    e1 = c1 / a1
    e2 = c2 / (a1 ** 2 + a2)
    with np.errstate(divide="ignore", invalid="ignore"):
        d_stdev = np.sqrt((e1 * S) + (e2 * S * (S - 1)))
        return S, n, theta_hat_w_abs, d / d_stdev


def close(a, b, tol=1e-12):
    """Equal NaN pattern, and within tol relative (absolute below 1)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    nan = np.isnan(b)
    if not np.array_equal(np.isnan(a), nan):
        return False
    return bool(np.all(np.abs(a[~nan] - b[~nan]) <= tol * np.maximum(1.0, np.abs(b[~nan]))))


# ------------------------------------------------------------------------------------------- CPU: the restatement itself
def test_restatement_matches_scikit_allel_tajima_d():
    rng = np.random.default_rng(21)
    for trial in range(12):
        S = int(rng.integers(300, 3000))
        ns = rng.integers(1, 60, size=2)
        cnt = np.zeros((S, 4), np.int64)
        for i in range(2):  # variable n: each row calls a random subset of 2 ns alleles; some rows are rare variants
            n = rng.binomial(2 * ns[i], rng.uniform(0.3, 1.0, S))
            p = np.where(rng.random(S) < 0.3, 1.0 / np.maximum(2 * ns[i], 1), rng.uniform(0, 1, S))
            a = rng.binomial(n, p)
            cnt[:, 2 * i], cnt[:, 2 * i + 1] = n - a, a
        pos = np.sort(rng.choice(np.arange(1, 40 * S), size=S, replace=False)).astype(np.int64)
        off = np.array([0, S // 3, S])
        flags = np.where(rng.random(S) < 0.1, 2, 3).astype(np.uint8)
        size = int(rng.choice([500, 5000, 20000]))
        r = restate(cnt, pos, off, size, flags=flags)
        wins = candidate_windows(pos, off, size, False)
        checked = 0
        for w, (_, lo, hi, _, _) in enumerate(wins):
            rows = np.arange(lo, hi)[(flags[lo:hi] & 1) != 0]
            for i, p in ((0, "_p1"), (1, "_p2")):
                if len(rows) == 0:
                    assert r["n_max" + p][w] == 0 and np.isnan(r["theta_w" + p][w]) and r["n_seg" + p][w] == 0
                    continue
                Sk, nk, twk, dk = skallel_tajima_d(cnt[rows][:, 2 * i:2 * i + 2])
                assert r["n_seg" + p][w] == Sk and r["n_max" + p][w] == nk, (trial, w, i)
                assert close(r["theta_w" + p][w], twk if nk >= 2 else np.nan), (trial, w, i)
                assert close(r["tajima_d" + p][w], dk if np.isfinite(dk) else np.nan), (trial, w, i)
                checked += np.isfinite(dk)
        assert checked > 0


def test_restatement_known_cases():
    def one(rows, flags=None):
        return restate(np.array(rows), np.arange(1, len(rows) + 1), [0, len(rows)], 10 ** 6, flags=flags)

    # n = 4: 8 singletons and 3 doubletons -> theta_pi = 8/2 + 3 * 2/3 = 6 = 11 / a1(4) = theta_w, D = 0
    r = one([[3, 1, 2, 2]] * 8 + [[2, 2, 2, 2]] * 3)
    assert r["n_seg_p1"][0] == 11 and r["n_max_p1"][0] == 4
    assert abs(r["theta_pi_p1"][0] - 6) <= 1e-12 and abs(r["theta_w_p1"][0] - 6) <= 1e-12
    assert abs(r["tajima_d_p1"][0]) <= 1e-12
    # Tajima's constants at n = 10
    a1t, a2t = harmonic_tables(10)
    e1, e2 = tajima_constants(10, a1t[10], a2t[10])
    assert abs(e1 - 0.019060533801591818) <= 1e-15 and abs(e2 - 0.00494892776989633) <= 1e-15
    # all singletons: an excess of rare variants
    r = one([[9, 1, 5, 5]] * 20)
    assert r["tajima_d_p1"][0] < 0 and r["tajima_d_p2"][0] > 0
    # fewer than 3 segregating sites: D undefined, theta_w defined
    r = one([[9, 1, 5, 5], [10, 0, 5, 5]])
    assert r["n_seg_p1"][0] == 1 and np.isnan(r["tajima_d_p1"][0]) and np.isfinite(r["theta_w_p1"][0])
    # n_max = 2 with S >= 3: e1 = e2 = 0, D undefined
    r = one([[1, 1, 5, 5]] * 4)
    assert r["n_seg_p1"][0] == 4 and r["n_max_p1"][0] == 2 and np.isnan(r["tajima_d_p1"][0])
    # no row passes the filters: n_max 0, theta_w undefined
    r = one([[3, 2, 4, 1]] * 4, flags=np.array([2, 2, 2, 2], np.uint8))
    assert r["n_max_p1"][0] == 0 and np.isnan(r["theta_w_p1"][0]) and r["snp_count"][0] == 4 and r["theta_pi_p1"][0] == 0
    # a row uncalled in the other population still counts toward S (and theta_pi)
    r = one([[2, 3, 0, 0], [4, 1, 1, 0]])
    assert r["n_seg_p1"][0] == 2 and r["n_seg_p2"][0] == 0 and r["n_max_p2"][0] == 1
    assert abs(r["theta_pi_p1"][0] - 1.0) <= 1e-15 and np.isnan(r["theta_w_p2"][0])


def test_save_csv_stats_tajima_columns(tmp_path):
    import twoDSFS_class as K
    stats = {"c1 1-100": {"snp_count": 3, "T2D": 1.5, "T1D_pop1": None, "T1D_pop2": 0.25, "new_term_pop1": 1.0,
                          "new_term_pop2": 1.25, "T2D_diff": None},
             "c1 101-200": {"snp_count": 1, "T2D": 2.0, "T1D_pop1": 0.5, "T1D_pop2": 0.5, "new_term_pop1": 1.5,
                            "new_term_pop2": 1.5, "T2D_diff": 1.5},
             "c2 1-100": {"snp_count": 2, "T2D": 0.0, "T1D_pop1": 0.0, "T1D_pop2": 0.0, "new_term_pop1": 0.0,
                          "new_term_pop2": 0.0, "T2D_diff": 0.0}}
    fst = {"c1 1-100": {"FST": 0.125}}
    taj = {"c1 1-100": {"TajimaD_pop1": -1.5, "TajimaD_pop2": None}, "c1 101-200": {"TajimaD_pop1": 0.75, "TajimaD_pop2": 2.0}}
    header = "chromosome,window_start,window_end,snp_count,T2D,T1D_p1,T1D_p2,new_term_p1,new_term_p2,T2D_diff"
    body = ["c1,1,100,3,1.5,,0.25,1.0,1.25,", "c1,101,200,1,2.0,0.5,0.5,1.5,1.5,1.5", "c2,1,100,2,0.0,0.0,0.0,0.0,0.0,0.0"]
    plain = tmp_path / "plain.csv"
    K.save_csv_stats(stats, str(plain))
    assert plain.read_bytes() == ("\r\n".join([header] + body) + "\r\n").encode()
    tail = [["-1.5", ""], ["0.75", "2.0"], ["", ""]]
    for kw, extra, cols in ((dict(tajima=taj), [], tail),
                            (dict(fst=fst, tajima=taj), ["FST"], [[f] + t for f, t in zip(["0.125", "", ""], tail)])):
        path = tmp_path / "t.csv"
        K.save_csv_stats(stats, str(path), **kw)
        rows = list(csv.reader(open(path, newline="")))
        assert rows[0] == header.split(",") + extra + ["TajimaD_p1", "TajimaD_p2"]
        assert [r[10:] for r in rows[1:]] == cols
        assert [r[:10] for r in rows[1:]] == [b.split(",") for b in body]


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


def assert_matches(res, exp, what=""):
    """GPU arrays per candidate window vs the restatement: labels and integers exact, theta and D to 1e-12."""
    n = len(exp["start"])
    assert len(res["start"]) == n, (what, len(res["start"]), n)
    for k in INTS:
        assert np.array_equal(res[k], exp[k]), (what, k)
    assert np.array_equal((res["flags"] & 8) != 0, exp["empty"]), what
    for k in FLOATS:
        assert close(res[k], exp[k]), (what, k)


@pytest.mark.gpu
@pytest.mark.parametrize("ns1,ns2,S,C,L", [
    (200, 200, 40000, 4, 400000),    # 14 + 14 words (compile-time instantiation)
    (500, 500, 12000, 3, 120000),    # 32 + 32 words (compile-time instantiation)
    (100, 37, 20000, 5, 200000),     # 8 + 4 words: runtime word count, uneven split
    (2100, 2100, 4000, 2, 60000),    # 132 + 132 words: rows wider than 4096 samples
])
def test_genotype_panels_vs_restatement_and_counts_entry(T, h, ns1, ns2, S, C, L):
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(ns1 * 7 + ns2 + S)
    c1, c2 = random_codes(rng, S, ns1, ns2)
    pos, off = random_positions(rng, S, C, L)
    G, w1, w2 = pack_codes(c1, c2)
    cnt = codes_to_counts(c1, c2)
    h.set_panel(ns1, ns2, True)
    defined = 0
    for size, snp in ((20000, False), (3000, False), (250, True), (1500, True)):
        h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
        a = h.neutrality(size, snp_mode=snp)
        exp = restate(cnt, pos, off, size, snp)
        assert_matches(a, exp, f"genotype {size} {snp}")
        defined += int(np.isfinite(a["tajima_d_p1"]).sum())
        h.load_counts(cnt.astype(np.uint16), pos, off)
        assert_bitwise(h.neutrality(size, snp_mode=snp), a, f"counts entry {size} {snp}")
    assert defined > 0


@pytest.mark.gpu
@pytest.mark.parametrize("tag,size,snp", [("20kb", 20000, False), ("500kb", 500000, False), ("500snps", 500, True)])
def test_chr1_golden_dict_tajima_scan(tag, size, snp):
    import twoDSFS_class as K
    from tdsfs_engine import SnpTable
    d = load_chr1_dict()
    inst = K.LikelihoodInference_jointSFS("x", "y")
    got = inst.tajima_scan_bySNPs(d, size) if snp else inst.tajima_scan(d, size)
    fst = inst.fst_scan_bySNPs(d, size) if snp else inst.fst_scan(d, size)
    assert list(got) == list(fst)
    t = SnpTable.from_dict(d, "uv", "bv")
    exp = restate(t.cnt, t.pos, t.off, size, snp)
    live = ~exp["empty"]
    keys = [f"{t.chroms[c]} {s}-{e}" for c, s, e in zip(exp["chrom"][live], exp["start"][live], exp["end"][live])]
    assert list(got) == keys
    names = K.LikelihoodInference_jointSFS._TAJIMA_COLS
    for i, k in enumerate(np.flatnonzero(live)):
        g = got[keys[i]]
        assert list(g) == list(names)
        for out, col in names.items():
            e = exp[col][k]
            if col in FLOATS:
                assert (g[out] is None) == bool(np.isnan(e)), (keys[i], out)
                assert g[out] is None or abs(g[out] - e) <= 1e-12 * max(1.0, abs(e)), (keys[i], out)
            else:
                assert g[out] == e, (keys[i], out)
    assert any(v["TajimaD_pop1"] is not None for v in got.values())


@pytest.mark.gpu
def test_half_calls_packed_panel_equals_dict_and_filters():
    import twoDSFS_class as K
    from tdsfs_engine import SnpTable, filter_flags
    vcf, pm = os.path.join(GOLDEN, "ingest_small.vcf.gz"), os.path.join(GOLDEN, "ingest_small.popmap.txt")
    inst = K.LikelihoodInference_jointSFS(vcf, pm, pop1_size=3, pop2_size=3)
    d, P = inst.make_data_dict_vcf(vcf, pm), inst.make_packed_panel()
    assert P.fixups is not None and len(P.fixups) > 0
    t = SnpTable.from_dict(d, "uv", "bv")
    for size, snp in ((30, False), (2, True)):
        fd = inst.tajima_scan_bySNPs(d, size) if snp else inst.tajima_scan(d, size)
        eng = inst._eng()
        a = eng.h.fetch_neutrality(eng.h.candidates(size, snp))
        fp = inst.tajima_scan_bySNPs(P, size) if snp else inst.tajima_scan(P, size)
        b = eng.h.fetch_neutrality(eng.h.candidates(size, snp))
        assert fd == fp
        assert_bitwise(a, b, f"ingest_small {size}")
        assert_matches(a, restate(t.cnt, t.pos, t.off, size, snp), f"ingest_small {size}")
    # constructor filters: chr1 with a variant type and a position range
    d = load_chr1_dict()
    t = SnpTable.from_dict(d, "uv", "bv")
    for ctor in (dict(variant_type="missense_variant"), dict(start_position=2_000_000, end_position=9_000_000),
                 dict(variant_type="intron_variant", start_position=5_000_000)):
        inst = K.LikelihoodInference_jointSFS("x", "y", **ctor)
        got = inst.tajima_scan(d, 100000)
        eng = inst._eng()
        res = eng.h.fetch_neutrality(eng.h.candidates(100000))
        flags = filter_flags(t, ctor.get("start_position"), ctor.get("end_position"), ctor.get("variant_type"))
        exp = restate(t.cnt, t.pos, t.off, 100000, False, flags)
        assert_matches(res, exp, str(ctor))
        whole = restate(t.cnt, t.pos, t.off, 100000, False)
        assert exp["n_seg_p1"].sum() < whole["n_seg_p1"].sum()
        assert len(got) == int((~exp["empty"]).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("size,snp", [(20000, False), (700, True)])
def test_shards_equal_whole_bitwise(T, size, snp):
    import tdsfs_dist as D
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(78)
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
        whole = h.neutrality(size, snp_mode=snp)
        parts, gathered = [], []
        for pieces in plan:
            a, b = pieces[0].lo, pieces[-1].hi
            Gr, _, _ = pack_codes(c1[a:b], c2[a:b])
            h.load_genotypes(Gr, b - a, w1, w2, ns1, ns2, pos[a:b], D.local_offsets(pieces))
            parts.append(D.localize_results(h.neutrality(size, snp_mode=snp), pieces, pos, size, snp))
            gathered.append(D.sharded_neutrality(h, pieces, pos, size, None, snp_mode=snp))
        for got in (parts, gathered):
            cat = {k: np.concatenate([p[k] for p in got]) for k in whole}
            assert_bitwise(cat, whole, "shards")
    finally:
        h.close()


@pytest.mark.gpu
def test_theta_pi_equals_fst_pass_pi_where_every_row_is_called(T, h):
    """With n >= 2 in both populations on every row, theta_pi_p* and the FST pass's pi_p* are the same sums."""
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(31)
    S, ns1, ns2 = 30000, 200, 200
    c1, c2 = random_codes(rng, S, ns1, ns2)
    c1[:3] = 1  # random_codes leaves rows with fewer than two called alleles: call them
    c2[5] = 1
    pos, off = random_positions(rng, S, 3, 300000)
    cnt = codes_to_counts(c1, c2)
    assert (cnt[:, 0] + cnt[:, 1] >= 2).all() and (cnt[:, 2] + cnt[:, 3] >= 2).all()
    G, w1, w2 = pack_codes(c1, c2)
    h.set_panel(ns1, ns2, True)
    h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
    for size, snp in ((20000, False), (2500, True)):
        n = h.neutrality(size, snp_mode=snp)
        d = h.diversity(size, snp_mode=snp)
        for i in ("1", "2"):
            assert np.array_equal(n["theta_pi_p" + i].view(np.uint64), d["pi_p" + i].view(np.uint64)), (size, i)


@pytest.mark.gpu
def test_neutrality_does_not_disturb_the_scan_or_the_fst_pass(T):
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(6)
    S, ns1, ns2, W = 30000, 200, 200, 20000
    c1, c2 = random_codes(rng, S, ns1, ns2)
    pos, off = random_positions(rng, S, 3, 300000)
    G, w1, w2 = pack_codes(c1, c2)

    def run(with_neut):
        h = T.Handle(0)
        try:
            h.set_panel(ns1, ns2, True)
            h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
            if with_neut:
                h.neutrality(5000, fetch=False)
            h.plan(W)
            if with_neut:
                h.neutrality(W, fetch=False)
            h.background(T.BG_GENOME)
            h.diversity(7000, fetch=False)
            if with_neut:
                h.neutrality(900, snp_mode=True, fetch=False)
            h.finalize_background()
            res = h.scan(W)
            fused = h.scan_info()[0]
            div = h.fetch_diversity(h.candidates(7000))
            steps, divs = [], []
            h.set_sync(False)
            for _ in range(3):
                h.step_bp(T.BG_GENOME, W)
                if with_neut:
                    h.neutrality(3000, snp_mode=True, fetch=False)
                h.diversity(W, fetch=False)
                if with_neut:
                    h.neutrality(W, fetch=False)
                h.check()
                steps.append(h.fetch_results(h.candidates(W)))
                divs.append(h.fetch_diversity(h.candidates(W)))
            h.set_sync(True)
            return res, fused, div, steps, divs
        finally:
            h.close()

    a, fa, da, sa, xa = run(True)
    b, fb, db, sb, xb = run(False)
    assert fa and fb, "the planned scan must stay on the fused path"
    assert_bitwise(a, b, "scan")
    assert_bitwise(da, db, "diversity")
    for x, y in zip(sa + xa, sb + xb):
        assert_bitwise(x, y, "step / diversity")


@pytest.mark.gpu
def test_error_conventions(T, h):
    import ctypes as C
    with pytest.raises(T.TdsfsError) as e:
        h.neutrality(1000)
    assert e.value.code == T.ERR_STATE
    h.set_panel(5, 5, True)
    with pytest.raises(T.TdsfsError) as e:
        h.neutrality(1000)
    assert e.value.code == T.ERR_STATE
    with pytest.raises(T.TdsfsError) as e:
        h.fetch_neutrality(10)
    assert e.value.code == T.ERR_STATE
    cnt = np.array([[4, 6, 5, 5]] * 100, dtype=np.uint16)
    pos = np.arange(1, 101, dtype=np.int32) * 50
    h.load_counts(cnt, pos, [0, 100])
    for size in (0, -3):
        with pytest.raises(T.TdsfsError) as e:
            h.neutrality(size)
        assert e.value.code == T.ERR_ARG
    n = h.candidates(1000)
    arrs, r = h._alloc_neutrality(n)
    nw = C.c_int64()
    assert h._L.tdsfs_neutrality_bp(h._h, C.c_int64(1000), C.byref(r), C.c_int64(n - 1), C.byref(nw)) == T.ERR_ARG
    assert h._L.tdsfs_neutrality_bp(h._h, C.c_int64(1000), C.byref(r), C.c_int64(n), C.byref(nw)) == 0 and nw.value == n
    assert h.neutrality(1000, fetch=False) == n
    with pytest.raises(T.TdsfsError) as e:
        h.fetch_neutrality(n - 1)
    assert e.value.code == T.ERR_ARG
    # the FST pass has its own results: no diversity call yet
    with pytest.raises(T.TdsfsError) as e:
        h.fetch_diversity(n)
    assert e.value.code == T.ERR_STATE


@pytest.mark.gpu
def test_chunked_host_upload(T, monkeypatch):
    import torch
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(10)
    S, ns1, ns2 = 50000, 200, 200
    c1, c2 = random_codes(rng, S, ns1, ns2)
    pos, off = random_positions(rng, S, 3, 500000)
    G, w1, w2 = pack_codes(c1, c2)
    out = []
    for host in (True, False):
        if host:
            monkeypatch.setenv("TDSFS_UPLOAD_CHUNK_KB", "16")
        else:
            monkeypatch.delenv("TDSFS_UPLOAD_CHUNK_KB", raising=False)
        h = T.Handle(0)
        try:
            h.set_panel(ns1, ns2, True)
            src = G if host else torch.from_numpy(G.view(np.int32)).cuda()
            h.load_genotypes(src, S, w1, w2, ns1, ns2, pos, off)
            out.append(h.neutrality(20000))  # before any background: the call itself waits for the upload
        finally:
            h.close()
    assert_bitwise(out[0], out[1], "chunked upload")
    assert_matches(out[0], restate(codes_to_counts(c1, c2), pos, off, 20000), "chunked upload")


@pytest.mark.gpu
def test_counts_entry_largest_n_is_in_the_table(T, h):
    """A counts-entry row can hold ref = alt = 65535 (n = 131070): the a1 / a2 table reaches it."""
    rng = np.random.default_rng(4)
    S = 64
    cnt = rng.integers(0, 40, size=(S, 4)).astype(np.int64)
    cnt[10] = [65535, 65535, 65535, 65535]
    cnt[40] = [1, 70000 - 65535, 65535, 1]
    cnt = np.minimum(cnt, 65535)
    pos = np.arange(1, S + 1, dtype=np.int32) * 10
    h.set_panel(5, 5, True)
    h.load_counts(cnt.astype(np.uint16), pos, [0, S])
    for size in (1000, 300):
        res = h.neutrality(size)
        exp = restate(cnt, pos, [0, S], size)
        assert_matches(res, exp, f"n = 131070, size {size}")
        assert res["n_max_p1"].max() == 131070 and res["n_max_p2"].max() == 131070
        assert np.isfinite(res["tajima_d_p1"]).all()
