"""Per-window Hudson FST, pi and dxy (tdsfs_diversity_*, fst_scan): a numpy restatement of the definition in DESIGN.md
section 7, checked on the CPU against Bhatia et al.'s per-site estimator, then the GPU results against the restatement.

Definition: a SNP enters a window iff it passes the spectrum filters (snp_flags bit0) and n_i = ref_i + alt_i >= 2 in both
populations; pi_i = 2 ref_i alt_i / (n_i (n_i - 1)), dxy = (ref_1 alt_2 + alt_1 ref_2) / (n_1 n_2) per site (fp64, one
division each); the window sums run in segments of SEG rows from the window's first row, lane (s - lo) mod 32 adding its
SNPs in row order, an xor tree over the 32 lanes, segment sums in order; FST = 1 - (pi_1 + pi_2) / (2 dxy), NaN at dxy == 0."""
import csv
import os

import numpy as np
import pytest

from helpers import GOLDEN, load_chr1_dict

SEG = 1024
FIELDS = ("pi_p1", "pi_p2", "dxy")


# ------------------------------------------------------------------------------------------- restatement (numpy)
def site_terms(cnt, passes=None):
    """cnt[S, 4] = (ref1, alt1, ref2, alt2) after fix-ups -> (entered, terms[S, 3] = pi_1, pi_2, dxy; 0 where not entered)."""
    r1, a1, r2, a2 = (np.asarray(cnt, dtype=np.int64)[:, i] for i in range(4))
    n1, n2 = r1 + a1, r2 + a2
    enter = (n1 >= 2) & (n2 >= 2)
    if passes is not None:
        enter &= np.asarray(passes, dtype=bool)
    t = np.zeros((len(r1), 3))
    e = enter
    t[e, 0] = (2 * r1[e] * a1[e]).astype(np.float64) / (n1[e] * (n1[e] - 1)).astype(np.float64)
    t[e, 1] = (2 * r2[e] * a2[e]).astype(np.float64) / (n2[e] * (n2[e] - 1)).astype(np.float64)
    t[e, 2] = (r1[e] * a2[e] + a1[e] * r2[e]).astype(np.float64) / (n1[e] * n2[e]).astype(np.float64)
    return enter, t


def window_sums(terms, lo, hi, seg=SEG):
    """The sums of rows [lo, hi) in the defined order."""
    total = np.zeros(terms.shape[1])
    lane_idx = np.arange(32)
    for g0 in range(lo, hi, seg):
        g1 = min(g0 + seg, hi)
        lanes = np.zeros((32, terms.shape[1]))
        for b in range(g0, g1, 32):
            m = min(32, g1 - b)
            lanes[:m] = lanes[:m] + terms[b:b + m]
        for o in (16, 8, 4, 2, 1):
            lanes = lanes + lanes[lane_idx ^ o]
        total = total + lanes[0]
    return total


def candidate_windows(pos, off, size, snp_mode):
    """(chrom, lo, hi, start, end) of every candidate window, in scan order (fixed-bp: window k of a chromosome holds
    positions 1 + kW .. (k+1)W, position 0 in window 0; fixed-SNP: full chunks of N rows, labels as scan_perChr_bySNPs)."""
    out = []
    for c in range(len(off) - 1):
        a, b = int(off[c]), int(off[c + 1])
        if b == a:
            continue
        p = np.asarray(pos[a:b], dtype=np.int64)
        if snp_mode:
            for j in range((b - a) // size):
                lo, hi = a + j * size, a + (j + 1) * size
                out.append((c, lo, hi, int(p[0]) if j == 0 else int(pos[lo - 1]) + 1, int(pos[hi - 1])))
        else:
            k = np.maximum(p - 1, 0) // size
            for kk in range(int(k[-1]) + 1):
                lo, hi = a + int(np.searchsorted(k, kk, "left")), a + int(np.searchsorted(k, kk, "right"))
                out.append((c, lo, hi, 1 + kk * size, (kk + 1) * size))
    return out


def restate(cnt, pos, off, size, snp_mode=False, flags=None):
    """Arrays per candidate window, as tdsfs_diversity_* returns them."""
    passes = None if flags is None else (np.asarray(flags) & 1) != 0
    counted = np.ones(len(cnt), dtype=np.int64) if flags is None else (np.asarray(flags, dtype=np.int64) >> 1) & 1
    enter, t = site_terms(cnt, passes)
    wins = candidate_windows(pos, off, size, snp_mode)
    r = {k: [] for k in ("chrom", "start", "end", "snp_count", "n_sites", "pi_p1", "pi_p2", "dxy", "fst", "empty")}
    for c, lo, hi, st, en in wins:
        s = window_sums(t, lo, hi)
        r["chrom"].append(c); r["start"].append(st); r["end"].append(en); r["empty"].append(hi == lo)
        r["snp_count"].append(int(counted[lo:hi].sum())); r["n_sites"].append(int(enter[lo:hi].sum()))
        r["pi_p1"].append(s[0]); r["pi_p2"].append(s[1]); r["dxy"].append(s[2])
        r["fst"].append(np.nan if s[2] == 0 else 1.0 - (s[0] + s[1]) / (2.0 * s[2]))
    return {k: np.array(v) for k, v in r.items()}


def codes_to_counts(c1, c2):
    """(ref1, alt1, ref2, alt2) of 2-bit codes on the host: 0 = 0/0, 1 = 0/1, 3 = 1/1, 2 = missing."""
    def rc(c):
        return (c == 1).sum(1) + 2 * (c == 0).sum(1), (c == 1).sum(1) + 2 * (c == 3).sum(1)
    (r1, a1), (r2, a2) = rc(c1), rc(c2)
    return np.stack([r1, a1, r2, a2], axis=1).astype(np.int64)


# ------------------------------------------------------------------------------------------- CPU: the restatement itself
def test_restatement_matches_bhatia_per_site_estimator():
    """Per site, Bhatia et al. (2013) eq. 10: N = (p1-p2)^2 - p1(1-p1)/(n1-1) - p2(1-p2)/(n2-1), D = p1(1-p2) + p2(1-p1);
    Hudson's FST of a window is sum N / sum D, which must equal 1 - (pi_1 + pi_2) / (2 dxy) of the summed terms."""
    rng = np.random.default_rng(11)
    for _ in range(20):
        S = int(rng.integers(50, 3000))
        n1 = rng.integers(2, 80, size=S)
        n2 = rng.integers(2, 80, size=S)
        a1, a2 = rng.integers(0, n1 + 1), rng.integers(0, n2 + 1)
        cnt = np.stack([n1 - a1, a1, n2 - a2, a2], axis=1)
        enter, t = site_terms(cnt)
        assert enter.all()
        p1, p2 = a1 / n1, a2 / n2
        N = (p1 - p2) ** 2 - p1 * (1 - p1) / (n1 - 1) - p2 * (1 - p2) / (n2 - 1)
        D = p1 * (1 - p2) + p2 * (1 - p1)
        assert np.allclose(t[:, 2], D, rtol=1e-12, atol=1e-15)
        assert np.allclose(t[:, 2] - (t[:, 0] + t[:, 1]) / 2, N, rtol=1e-12, atol=1e-14)
        s = window_sums(t, 0, S)
        if D.sum() > 0:
            assert abs((1 - (s[0] + s[1]) / (2 * s[2])) - N.sum() / D.sum()) <= 1e-12 * max(1.0, abs(N.sum() / D.sum()))


def test_restatement_known_cases():
    # a fixed difference: FST = 1
    r = restate(np.array([[10, 0, 0, 8]] * 5), np.arange(1, 6), [0, 5], 100)
    assert r["n_sites"][0] == 5 and r["fst"][0] == 1.0 and r["pi_p1"][0] == 0 and r["dxy"][0] == 5.0
    # no SNP passes the filters: n_sites 0, FST undefined
    r = restate(np.array([[3, 2, 4, 1]] * 4), np.arange(1, 5), [0, 4], 100, flags=np.array([2, 2, 2, 2], np.uint8))
    assert r["n_sites"][0] == 0 and np.isnan(r["fst"][0]) and r["snp_count"][0] == 4
    # a site with fewer than two called alleles in a population is excluded
    r = restate(np.array([[1, 0, 3, 3], [2, 2, 1, 0], [2, 2, 3, 3]]), np.array([1, 2, 3]), [0, 3], 100)
    assert r["n_sites"][0] == 1 and r["dxy"][0] == 0.5
    # equal sample frequencies: Hudson's FST is negative (the within-population terms carry the n / (n - 1) correction)
    r = restate(np.array([[5, 5, 5, 5], [6, 2, 6, 2]]), np.array([1, 2]), [0, 2], 100)
    assert r["fst"][0] < 0


def test_restatement_segments_and_lanes():
    """Windows longer than one segment and starting mid-block sum to the plain sum up to rounding."""
    rng = np.random.default_rng(3)
    cnt = np.stack([rng.integers(0, 20, 5000), rng.integers(0, 20, 5000), rng.integers(0, 20, 5000), rng.integers(0, 20, 5000)], 1)
    _, t = site_terms(cnt)
    s = window_sums(t, 37, 4321)
    assert np.allclose(s, t[37:4321].sum(0), rtol=1e-12)


def test_save_csv_stats_fst_column(tmp_path):
    import twoDSFS_class as K
    stats = {"c1 1-100": {"snp_count": 3, "T2D": 1.5, "T1D_pop1": None, "T1D_pop2": 0.25, "new_term_pop1": 1.0,
                          "new_term_pop2": 1.25, "T2D_diff": None},
             "c1 101-200": {"snp_count": 1, "T2D": 2.0, "T1D_pop1": 0.5, "T1D_pop2": 0.5, "new_term_pop1": 1.5,
                            "new_term_pop2": 1.5, "T2D_diff": 1.5},
             "c2 1-100": {"snp_count": 2, "T2D": 0.0, "T1D_pop1": 0.0, "T1D_pop2": 0.0, "new_term_pop1": 0.0,
                          "new_term_pop2": 0.0, "T2D_diff": 0.0}}
    fst = {"c1 1-100": {"FST": 0.125}, "c1 101-200": {"FST": None}}
    plain, with_fst = tmp_path / "plain.csv", tmp_path / "fst.csv"
    K.save_csv_stats(stats, str(plain))
    K.save_csv_stats(stats, str(with_fst), fst=fst)
    header = "chromosome,window_start,window_end,snp_count,T2D,T1D_p1,T1D_p2,new_term_p1,new_term_p2,T2D_diff"
    body = ["c1,1,100,3,1.5,,0.25,1.0,1.25,", "c1,101,200,1,2.0,0.5,0.5,1.5,1.5,1.5", "c2,1,100,2,0.0,0.0,0.0,0.0,0.0,0.0"]
    assert plain.read_bytes() == ("\r\n".join([header] + body) + "\r\n").encode()
    rows = list(csv.reader(open(with_fst, newline="")))
    assert rows[0] == header.split(",") + ["FST"]
    assert [r[-1] for r in rows[1:]] == ["0.125", "", ""]
    assert [r[:-1] for r in rows[1:]] == [b.split(",") for b in body]


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
    """GPU arrays per candidate window vs the restatement: labels and counts exact, sums to 1e-12 relative."""
    n = len(exp["start"])
    assert len(res["start"]) == n, (what, len(res["start"]), n)
    for k in ("chrom", "start", "end", "snp_count", "n_sites"):
        assert np.array_equal(res[k], exp[k]), (what, k)
    assert np.array_equal((res["flags"] & 8) != 0, exp["empty"]), what
    for k in FIELDS:
        err = np.abs(res[k] - exp[k]) / np.maximum(np.abs(exp[k]), 1e-300)
        assert n == 0 or err.max() <= 1e-12, (what, k, err.max())
    nan = np.isnan(exp["fst"])
    assert np.array_equal(np.isnan(res["fst"]), nan), what
    assert np.all(np.abs(res["fst"][~nan] - exp["fst"][~nan]) <= 1e-12 * np.maximum(1.0, np.abs(exp["fst"][~nan]))), what


def assert_bitwise(a, b, what=""):
    assert list(a) == list(b)
    for k in a:
        assert a[k].dtype == b[k].dtype and np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), (what, k)


def random_codes(rng, S, ns1, ns2, miss=0.04):
    f = np.exp(rng.uniform(np.log(0.003), np.log(0.997), size=S))

    def codes(ns):
        p = np.clip(f + rng.normal(0, 0.08, S) * np.sqrt(f * (1 - f)), 0, 1)[:, None]
        a = (rng.random((S, ns)) < p).astype(np.uint8) + (rng.random((S, ns)) < p).astype(np.uint8)
        c = np.where(a == 2, 3, a).astype(np.uint8)
        c[rng.random((S, ns)) < miss] = 2
        return c

    c1, c2 = codes(ns1), codes(ns2)
    c1[:3] = 2  # a few SNPs with no called allele in population 1: excluded
    c2[5, :] = 2
    c2[5, 0] = 1
    return c1, c2


def random_positions(rng, S, C, L):
    sizes = rng.multinomial(S, np.ones(C) / C)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    # the last chromosome is spread over a 20x longer stretch: many empty windows
    pos = np.concatenate([np.sort(rng.choice(np.arange(0, L * (20 if c == C - 1 else 1)), size=s, replace=False))
                          for c, s in enumerate(sizes)]).astype(np.int32)
    return pos, off


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
    longest = 0
    for size, snp in ((20000, False), (3000, False), (250, True), (1500, True)):
        h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
        a = h.diversity(size, snp_mode=snp)
        exp = restate(cnt, pos, off, size, snp)
        assert_matches(a, exp, f"genotype {size} {snp}")
        if not snp and size == 3000:
            assert (a["flags"] & T.F_EMPTY).any(), "the panel must have empty windows"
        longest = max(longest, int(a["snp_count"].max()))
        h.load_counts(cnt.astype(np.uint16), pos, off)
        assert_bitwise(h.diversity(size, snp_mode=snp), a, f"counts entry {size} {snp}")
    assert longest > SEG, "some window must span more than one segment"


@pytest.mark.gpu
@pytest.mark.parametrize("tag,size,snp", [("20kb", 20000, False), ("500kb", 500000, False), ("500snps", 500, True)])
def test_chr1_golden_dict_fst_scan(tag, size, snp):
    import twoDSFS_class as K
    from tdsfs_engine import SnpTable
    d = load_chr1_dict()
    inst = K.LikelihoodInference_jointSFS("x", "y")
    got = inst.fst_scan_bySNPs(d, size) if snp else inst.fst_scan(d, size)
    if snp:
        assert set(inst.scan_perChr_bySNPs(d, size)) <= set(got)
    else:
        assert list(inst.combined_scan(d, size)) == list(got)
    t = SnpTable.from_dict(d, "uv", "bv")
    exp = restate(t.cnt, t.pos, t.off, size, snp)
    live = ~exp["empty"]
    keys = [f"{t.chroms[c]} {s}-{e}" for c, s, e in zip(exp["chrom"][live], exp["start"][live], exp["end"][live])]
    assert list(got) == keys
    for i, k in enumerate(np.flatnonzero(live)):
        g = got[keys[i]]
        assert g["snp_count"] == exp["snp_count"][k] and g["n_sites"] == exp["n_sites"][k]
        for f, e in (("pi_pop1", "pi_p1"), ("pi_pop2", "pi_p2"), ("dxy", "dxy")):
            assert abs(g[f] - exp[e][k]) <= 1e-12 * abs(exp[e][k]), (keys[i], f)
        if np.isnan(exp["fst"][k]):
            assert g["FST"] is None
        else:
            assert abs(g["FST"] - exp["fst"][k]) <= 1e-12 * max(1.0, abs(exp["fst"][k]))


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
        fd = inst.fst_scan_bySNPs(d, size) if snp else inst.fst_scan(d, size)
        eng = inst._eng()
        a = eng.h.fetch_diversity(eng.h.candidates(size, snp))
        fp = inst.fst_scan_bySNPs(P, size) if snp else inst.fst_scan(P, size)
        b = eng.h.fetch_diversity(eng.h.candidates(size, snp))
        assert fd == fp
        assert_bitwise(a, b, f"ingest_small {size}")
        assert_matches(a, restate(t.cnt, t.pos, t.off, size, snp), f"ingest_small {size}")
    # constructor filters: chr1 with a variant type and a position range
    d = load_chr1_dict()
    t = SnpTable.from_dict(d, "uv", "bv")
    for ctor in (dict(variant_type="missense_variant"), dict(start_position=2_000_000, end_position=9_000_000),
                 dict(variant_type="intron_variant", start_position=5_000_000)):
        inst = K.LikelihoodInference_jointSFS("x", "y", **ctor)
        got = inst.fst_scan(d, 100000)
        eng = inst._eng()
        res = eng.h.fetch_diversity(eng.h.candidates(100000))
        flags = filter_flags(t, ctor.get("start_position"), ctor.get("end_position"), ctor.get("variant_type"))
        exp = restate(t.cnt, t.pos, t.off, 100000, False, flags)
        assert_matches(res, exp, str(ctor))
        whole = restate(t.cnt, t.pos, t.off, 100000, False)
        assert exp["n_sites"].sum() < whole["n_sites"].sum()
        assert len(got) == int((~exp["empty"]).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("size,snp", [(20000, False), (700, True)])
def test_shards_equal_whole_bitwise(T, size, snp):
    import tdsfs_dist as D
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(77)
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
        whole = h.diversity(size, snp_mode=snp)
        parts, gathered = [], []
        for pieces in plan:
            a, b = pieces[0].lo, pieces[-1].hi
            Gr, _, _ = pack_codes(c1[a:b], c2[a:b])
            h.load_genotypes(Gr, b - a, w1, w2, ns1, ns2, pos[a:b], D.local_offsets(pieces))
            parts.append(D.localize_results(h.diversity(size, snp_mode=snp), pieces, pos, size, snp))
            gathered.append(D.sharded_diversity(h, pieces, pos, size, None, snp_mode=snp))
        for got in (parts, gathered):
            cat = {k: np.concatenate([p[k] for p in got]) for k in whole}
            assert_bitwise(cat, whole, "shards")
    finally:
        h.close()


@pytest.mark.gpu
def test_diversity_does_not_disturb_the_scan(T):
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(5)
    S, ns1, ns2, W = 30000, 200, 200, 20000
    c1, c2 = random_codes(rng, S, ns1, ns2)
    pos, off = random_positions(rng, S, 3, 300000)
    G, w1, w2 = pack_codes(c1, c2)

    def run(with_div):
        h = T.Handle(0)
        try:
            h.set_panel(ns1, ns2, True)
            h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
            h.plan(W)
            h.background(T.BG_GENOME)
            if with_div:
                h.diversity(7000, fetch=False)
            h.finalize_background()
            res = h.scan(W)
            fused = h.scan_info()[0]
            steps = []
            for _ in range(3):
                h.step_bp(T.BG_GENOME, W)
                if with_div:
                    h.diversity(3000, snp_mode=True, fetch=False)
                    h.diversity(7000)
                h.check()
                steps.append(h.fetch_results(h.candidates(W)))
            return res, fused, steps
        finally:
            h.close()

    a, fa, sa = run(True)
    b, fb, sb = run(False)
    assert fa and fb, "the planned scan must stay on the fused path"
    assert_bitwise(a, b, "scan")
    for x, y in zip(sa, sb):
        assert_bitwise(x, y, "step")


@pytest.mark.gpu
def test_error_conventions(T, h):
    import ctypes as C
    with pytest.raises(T.TdsfsError) as e:
        h.diversity(1000)
    assert e.value.code == T.ERR_STATE
    h.set_panel(5, 5, True)
    with pytest.raises(T.TdsfsError) as e:
        h.diversity(1000)
    assert e.value.code == T.ERR_STATE
    with pytest.raises(T.TdsfsError) as e:
        h.fetch_diversity(10)
    assert e.value.code == T.ERR_STATE
    cnt = np.array([[4, 6, 5, 5]] * 100, dtype=np.uint16)
    pos = np.arange(1, 101, dtype=np.int32) * 50
    h.load_counts(cnt, pos, [0, 100])
    for size in (0, -3):
        with pytest.raises(T.TdsfsError) as e:
            h.diversity(size)
        assert e.value.code == T.ERR_ARG
    n = h.candidates(1000)
    arrs, r = h._alloc_diversity(n)
    nw = C.c_int64()
    assert h._L.tdsfs_diversity_bp(h._h, C.c_int64(1000), C.byref(r), C.c_int64(n - 1), C.byref(nw)) == T.ERR_ARG
    assert h._L.tdsfs_diversity_bp(h._h, C.c_int64(1000), C.byref(r), C.c_int64(n), C.byref(nw)) == 0 and nw.value == n
    assert h.diversity(1000, fetch=False) == n
    with pytest.raises(T.TdsfsError) as e:
        h.fetch_diversity(n - 1)
    assert e.value.code == T.ERR_ARG


@pytest.mark.gpu
def test_chunked_host_upload(T, monkeypatch):
    import torch
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(9)
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
            out.append(h.diversity(20000))  # before any background: the call itself waits for the upload
        finally:
            h.close()
    assert_bitwise(out[0], out[1], "chunked upload")
    assert_matches(out[0], restate(codes_to_counts(c1, c2), pos, off, 20000), "chunked upload")
