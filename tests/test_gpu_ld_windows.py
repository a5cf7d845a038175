"""Per-window linkage disequilibrium, Kelly's ZnS and Kim and Nielsen's omega (tdsfs_ld_windows_*, ld_scan): a numpy /
Python-int restatement of the definition in DESIGN.md section 7, checked on the CPU against a literal restatement of
scikit-allel's pairwise r (gn_pairwise_corrcoef_int8) and a brute-force Kim and Nielsen omega, then the GPU results
against the restatement, bit for bit.

Definition, per window and population over the window's rows that pass the spectrum filter and that population's samples
(codes 0, 1, 3 = dosage 0, 1, 2; code 2 missing, fix-up calls included): a site is a row whose called dosages are not all
equal; a pair i < j is defined iff vx vy > 0 over the samples called in both (r^2 as in LD pruning), and enters as
q = rint(2^32 r^2).  zns = 2^-32 sum q / n_pairs; omega = max over splits 2 <= k <= m - 2 of the sites of
((WL + WR) / (nL + nR)) / (X / nX) with nL + nR > 0 and X > 0, the lowest k on ties."""
import csv
import os

import numpy as np
import pytest

from helpers import GOLDEN
from test_gpu_diversity import assert_bitwise, candidate_windows, random_codes, random_positions
from test_gpu_ldprune import DOSE, ld_rich_codes, pair_sums, r2_exact, skallel_corrcoef

INTS = ("chrom", "start", "end", "snp_count", "n_sites_p1", "n_sites_p2", "n_pairs_p1", "n_pairs_p2", "omega_pos_p1",
        "omega_pos_p2")
FLOATS = ("zns_p1", "zns_p2", "omega_p1", "omega_p2")
F32_TOL = 2.0 ** -17  # scikit-allel's r^2 from float32 moments: E[xy] - E[x] E[y] cancels at a few 2^-24 of E[xy] <= 4


# ------------------------------------------------------------------------------------------- restatement
def pair_matrices(x):
    """(n, Sx, Sy, Qx, Qy, P) as int64 [R, R] matrices ([i, j]: rows i and j over the samples called in both) of dosages
    x [R, ns] (-1 missing), from fp64 products of small integers (exact)."""
    c = (x >= 0).astype(np.float64)
    v = np.where(x >= 0, x, 0).astype(np.float64)
    v2 = v * v
    return tuple(np.rint(m).astype(np.int64) for m in (c @ c.T, v @ c.T, c @ v.T, v2 @ c.T, c @ v2.T, v @ v.T))


def window_ld(x, splits=False):
    """One window and population, dosages x [R, ns] of its rows in order: (m, n_pairs, sum q, zns, omega, row of s_k at the
    best split or -1) and, with splits, the list of (k, omega_k) of the eligible splits.  Integer sums are Python ints."""
    R = len(x)
    if R == 0:
        out = (0, 0, 0, np.nan, np.nan, -1)
        return out + ([],) if splits else out
    n, Sx, Sy, Qx, Qy, P = pair_matrices(x)
    site = np.diag(n * Qx - Sx * Sx) > 0
    r2 = r2_exact(n, Sx, Sy, Qx, Qy, P)
    defined = np.isfinite(r2) & np.triu(np.ones((R, R), bool), 1)
    q = np.where(defined, np.rint(np.where(defined, r2, 0.0) * 2.0 ** 32), 0.0).astype(np.uint64)
    assert int(q.max(initial=0)) <= 2 ** 32 and R < 90000  # every uint64 sum below is exact
    T, N = int(q.sum()), int(defined.sum())
    zns = np.nan if N == 0 else float(T) * 2.0 ** -32 / float(N)
    WLc, Pd = np.cumsum(q.sum(0)), np.cumsum(q.sum(1))   # sums of c_j (pairs ending at j) and of d_i (pairs from i)
    nLc, nPd = np.cumsum(defined.sum(0)), np.cumsum(defined.sum(1))
    sites = np.flatnonzero(site)
    m = len(sites)
    best, best_row, eligible = -1.0, -1, []
    for k in range(2, m - 1):
        r = sites[k - 1]
        WL, Pk, nL, nP = int(WLc[r]), int(Pd[r]), int(nLc[r]), int(nPd[r])
        WR, X, nR, nX = T - Pk, Pk - WL, N - nP, nP - nL
        if nL + nR > 0 and X > 0:
            om = (float(WL + WR) / float(nL + nR)) / (float(X) / float(nX))
            eligible.append((k, om))
            if om > best:
                best, best_row = om, r
    out = (m, N, T, zns, best if best_row >= 0 else np.nan, best_row)
    return out + (eligible,) if splits else out


def restate(c1, c2, pos, off, size, snp_mode=False, flags=None):
    """Arrays per candidate window, as tdsfs_ld_windows_* returns them, from 2-bit codes [S, ns1], [S, ns2]."""
    S = len(c1)
    passes = np.ones(S, bool) if flags is None else (np.asarray(flags) & 1) != 0
    counted = np.ones(S, np.int64) if flags is None else (np.asarray(flags, dtype=np.int64) >> 1) & 1
    xs = (DOSE[np.asarray(c1, dtype=np.int64)], DOSE[np.asarray(c2, dtype=np.int64)])
    r = {k: [] for k in INTS + FLOATS + ("empty",)}
    for ch, lo, hi, st, en in candidate_windows(pos, off, size, snp_mode):
        rows = lo + np.flatnonzero(passes[lo:hi])
        r["chrom"].append(ch); r["start"].append(st); r["end"].append(en); r["empty"].append(hi == lo)
        r["snp_count"].append(int(counted[lo:hi].sum()))
        for p, x in enumerate(xs, 1):
            m, N, _, zns, om, row = window_ld(x[rows])
            r[f"n_sites_p{p}"].append(m); r[f"n_pairs_p{p}"].append(N); r[f"zns_p{p}"].append(zns)
            r[f"omega_p{p}"].append(om); r[f"omega_pos_p{p}"].append(int(pos[rows[row]]) if row >= 0 else -1)
    return {k: np.array(v, dtype=np.float64 if k in FLOATS else None) for k, v in r.items()}


def skallel_r2(x):
    """scikit-allel's rogers_huff_r ** 2 over rows x [R, ns] (gn_pairwise_corrcoef_int8, float32 throughout): the
    condensed pairs i < j in row order.  Vectorised statement of skallel_corrcoef, checked against it."""
    f = np.float32
    R = len(x)
    i, j = np.triu_indices(R, 1)
    a, b = x[i], x[j]
    both = (a >= 0) & (b >= 0)
    a, b = np.where(both, a, 0), np.where(both, b, 0)
    n = both.sum(1).astype(f)
    m0, m1, v0, v1, cov = (s.sum(1).astype(f) for s in (a, b, a * a, b * b, a * b))
    bad = (n == 0) | (v0 == 0) | (v1 == 0)
    with np.errstate(invalid="ignore", divide="ignore"):
        m0, m1, v0, v1, cov = m0 / n, m1 / n, v0 / n, v1 / n, cov / n
        cov = cov - m0 * m1
        v0 = v0 - m0 * m0
        v1 = v1 - m1 * m1
        r = (cov.astype(np.float64) / np.sqrt((v0 * v1).astype(np.float64))).astype(f)
    r[bad] = np.nan
    return r * r


def brute_omega(r2, sites):
    """Kim and Nielsen (2004) omega over the sites (all pairs defined), O(m^3): the largest
    [(sum_L + sum_R) / (C(k, 2) + C(m - k, 2))] / [sum_LR / (k (m - k))] over 2 <= k <= m - 2."""
    m = len(sites)
    best = np.nan
    for k in range(2, m - 1):
        L, R = sites[:k], sites[k:]
        wl = sum(r2[a, b] for x, a in enumerate(L) for b in L[x + 1:])
        wr = sum(r2[a, b] for x, a in enumerate(R) for b in R[x + 1:])
        xs = sum(r2[a, b] for a in L for b in R)
        if xs > 0:
            om = ((wl + wr) / (k * (k - 1) / 2 + (m - k) * (m - k - 1) / 2)) / (xs / (k * (m - k)))
            best = om if not best >= om else best
    return best


def codes_of(dose_rows):
    """Dosage rows (-1 missing) -> codes."""
    return np.array([0, 1, 3, 2])[np.asarray(dose_rows)].astype(np.uint8)


# ------------------------------------------------------------------------------------------- CPU: the restatement itself
def test_vectorised_skallel_equals_the_literal():
    rng = np.random.default_rng(5)
    c1, _ = ld_rich_codes(rng, 40, 17, 1, miss=0.2)
    x = DOSE[c1.astype(np.int64)]
    x[3] = 1                                  # all heterozygous: NaN
    got = skallel_r2(x)
    i, j = np.triu_indices(40, 1)
    want = np.array([np.float32(skallel_corrcoef(x[a], x[b])) ** 2 for a, b in zip(i, j)], dtype=np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("seed", range(4))
def test_restatement_matches_scikit_allel_and_brute_force(seed):
    rng = np.random.default_rng(40 + seed)
    S, ns1, ns2 = 240, 13 + seed, 9
    c1, c2 = ld_rich_codes(rng, S, ns1, ns2, miss=0.08)
    c1[10] = 1                                # all heterozygous in population 1
    pos = np.sort(rng.choice(np.arange(1, 30 * S), size=S, replace=False)).astype(np.int64)
    off = np.array([0, 100, S])
    flags = np.where(rng.random(S) < 0.1, 2, 3).astype(np.uint8)
    passes = (flags & 1) != 0
    size = 1500
    exp = restate(c1, c2, pos, off, size, flags=flags)
    checked = 0
    for w, (_, lo, hi, _, _) in enumerate(candidate_windows(pos, off, size, False)):
        rows = lo + np.flatnonzero(passes[lo:hi])
        for p, c in ((1, c1), (2, c2)):
            x = DOSE[c[rows].astype(np.int64)]
            r2 = skallel_r2(x).astype(np.float64)
            ok = np.isfinite(r2)
            assert exp[f"n_pairs_p{p}"][w] == int(ok.sum()), (w, p)
            if ok.any():
                # q rounds each r^2 by at most 2^-33; scikit-allel's float32 moments cancel in cov and v
                exact = r2_exact(*pair_matrices(x))[np.triu_indices(len(x), 1)]
                assert abs(exp[f"zns_p{p}"][w] - exact[ok].mean()) <= 2.0 ** -32, (w, p)
                assert abs(exp[f"zns_p{p}"][w] - r2[ok].mean()) <= F32_TOL + 2.0 ** -32, (w, p)
                checked += 1
            else:
                assert np.isnan(exp[f"zns_p{p}"][w])
    assert checked >= 10
    # without missing calls every pair of sites is defined: Kim and Nielsen's formula, O(m^3)
    c1, c2 = ld_rich_codes(rng, 60, 15, 11, miss=0.0)
    c1[[5, 17]] = 1
    for c in (c1, c2):
        x = DOSE[c.astype(np.int64)]
        m, N, _, _, om, row = window_ld(x)
        sums = pair_matrices(x)
        r2 = r2_exact(*sums)
        sites = np.flatnonzero(np.diag(sums[0] * sums[3] - sums[1] * sums[1]) > 0).tolist()
        assert len(sites) == m and N == m * (m - 1) // 2
        want = brute_omega(r2, sites)
        assert abs(om - want) <= 1e-8 * want and row in sites, (om, want)


def test_known_cases():
    rng = np.random.default_rng(0)
    A = rng.integers(0, 3, 24)
    A[:3] = [0, 1, 2]
    B = rng.integers(0, 3, 24)
    B[:3] = [2, 0, 1]

    def one(rows, splits=False):
        return window_ld(np.asarray(rows, dtype=np.int64), splits)

    # identical rows: ZnS = omega = 1 exactly, the first split (k = 2) wins the tie
    m, N, T, zns, om, row, sp = one([A] * 6, True)
    assert (m, N, T, zns, om, row) == (6, 15, 15 * 2 ** 32, 1.0, 1.0, 1) and [k for k, _ in sp] == [2, 3, 4]
    # two unlinked blocks: the best split is at the boundary
    assert one([A] * 5 + [B] * 6)[5] == 4
    rab = r2_exact(*pair_sums(np.array([A, B]), [0], [1]))[0]
    assert 0 < rab < 0.5
    # fewer than 4 sites: omega NaN; fewer than 2: no pair, ZnS NaN too
    m, N, _, zns, om, row = one([A, B, A])
    assert m == 3 and N == 3 and zns > 0 and np.isnan(om) and row == -1
    m, N, _, zns, om, row = one([A, np.ones(24, np.int64), np.full(24, -1)])
    assert m == 1 and N == 0 and np.isnan(zns) and np.isnan(om)
    # an all-heterozygous row is not a site and in no defined pair (Tajima's S would count it)
    het = np.ones(24, np.int64)
    assert one([A, het, A, B, het, B])[:2] == (4, 6)
    # two sites without a common call: no defined pair
    assert one([[0, 1, 2] + [-1] * 21, [-1] * 3 + [2, 0, 1] + [-1] * 18])[:2] == (2, 0)
    # a palindrome of rows gives omega_k = omega_{m-k} exactly: the lower k wins
    _, _, _, _, om, row, sp = one([A, A, B, B, A, A], True)
    d = dict(sp)
    assert d[2] == d[4] == om > d[3] and row == 1


def test_ld_scan_rejects_a_data_dict():
    import twoDSFS_class as K
    from helpers import rows_to_dict
    inst = K.LikelihoodInference_jointSFS("x", "y")
    d = rows_to_dict([["c1", 10, [3, 1], [2, 2], "No annotation"]], ("uv", "bv"))
    for call in (lambda: inst.ld_scan(d, 1000), lambda: inst.ld_scan_bySNPs(d, 10)):
        with pytest.raises(TypeError, match="make_packed_panel"):
            call()


def test_save_csv_stats_ld_columns(tmp_path):
    import twoDSFS_class as K
    stats = {"c1 1-100": {"snp_count": 3, "T2D": 1.5, "T1D_pop1": None, "T1D_pop2": 0.25, "new_term_pop1": 1.0,
                          "new_term_pop2": 1.25, "T2D_diff": None},
             "c2 1-100": {"snp_count": 2, "T2D": 0.0, "T1D_pop1": 0.0, "T1D_pop2": 0.0, "new_term_pop1": 0.0,
                          "new_term_pop2": 0.0, "T2D_diff": 0.0}}
    ld = {"c1 1-100": {"ZnS_pop1": 0.5, "ZnS_pop2": None, "omega_pop1": 2.25, "omega_pop2": None}}
    plain = tmp_path / "plain.csv"
    K.save_csv_stats(stats, str(plain), fst={"c1 1-100": {"FST": 0.1}})
    path = tmp_path / "ld.csv"
    K.save_csv_stats(stats, str(path), fst={"c1 1-100": {"FST": 0.1}}, tajima={}, ld=ld)
    rows = list(csv.reader(open(path, newline="")))
    assert rows[0][-7:] == ["FST", "TajimaD_p1", "TajimaD_p2", "ZnS_p1", "ZnS_p2", "omega_p1", "omega_p2"]
    assert rows[1][-4:] == ["0.5", "", "2.25", ""] and rows[2][-4:] == ["", "", "", ""]
    base = list(csv.reader(open(plain, newline="")))
    assert [r[:11] for r in rows] == base


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
    """GPU arrays per candidate window vs the restatement: every column bit for bit."""
    n = len(exp["start"])
    assert len(res["start"]) == n, (what, len(res["start"]), n)
    for k in INTS:
        assert np.array_equal(res[k], exp[k].astype(res[k].dtype)), (what, k, np.flatnonzero(res[k] != exp[k])[:5])
    assert np.array_equal((res["flags"] & 8) != 0, exp["empty"]), what
    for k in FLOATS:
        assert np.array_equal(res[k].view(np.uint64), exp[k].view(np.uint64)), (what, k)


def load(h, c1, c2, pos, off, flags=None, fixups=None):
    from tdsfs_pack import pack_codes
    ns1, ns2 = c1.shape[1], c2.shape[1]
    G, w1, w2 = pack_codes(c1, c2)
    h.set_panel(max(ns1, 2), max(ns2, 2), True)
    h.load_genotypes(G, len(c1), w1, w2, ns1, ns2, pos, off, fixups=fixups, flags=flags)


@pytest.mark.gpu
@pytest.mark.parametrize("ns1,ns2,S", [
    (500, 500, 3000),    # 32 + 32 words (compile-time instantiation)
    (200, 200, 4000),    # 14 + 14 words (compile-time instantiation)
    (33, 7, 5000),       # runtime word count, padding in both populations
    (1, 1, 5000),        # one sample per population
    (2100, 40, 1200),    # runtime, more word pairs than one staging pass holds, across the population boundary
])
def test_panels_vs_restatement(T, h, ns1, ns2, S):
    rng = np.random.default_rng(ns1 * 3 + ns2 + S)
    half = S // 2
    r1, r2 = random_codes(rng, S - half, ns1, ns2)
    l1, l2 = ld_rich_codes(rng, half, ns1, ns2)
    c1, c2 = np.concatenate([l1, r1]), np.concatenate([l2, r2])
    c1[rng.random(c1.shape) < 0.03] = 2
    c1[40] = 1                                   # all heterozygous: not a site
    # chromosome starts off the 32-row grid; positions dense enough for windows of more than 1024 rows
    off = np.array([0, 7, 1390 if S > 2000 else 390, S - 37, S], dtype=np.int64)
    pos = np.concatenate([np.sort(rng.choice(np.arange(1, 4 * (b - a) + 2), size=b - a, replace=False))
                          for a, b in zip(off[:-1], off[1:])]).astype(np.int32)
    flags = np.where(rng.random(S) < 0.1, 2, 3).astype(np.uint8)
    flags[rng.random(S) < 0.05] &= 1
    load(h, c1, c2, pos, off, flags=flags)
    defined = 0
    for size, snp in ((300, False), (5000, False), (97, True), (1500, True)):
        res = h.ld_windows(size, snp_mode=snp)
        assert_restated(res, restate(c1, c2, pos, off, size, snp, flags), f"{size} {snp}")
        defined += int(np.isfinite(res["omega_p1"]).sum() + np.isfinite(res["omega_p2"]).sum())
    assert defined > 10 or ns1 == 1
    assert h.ld_windows_ms() > 0


@pytest.mark.gpu
def test_empty_windows_and_no_flags(T, h):
    rng = np.random.default_rng(9)
    S = 2000
    c1, c2 = ld_rich_codes(rng, S, 20, 30)
    pos, off = random_positions(rng, S, 3, 40000)   # the last chromosome is sparse: many empty windows
    load(h, c1, c2, pos, off)
    for size, snp in ((1000, False), (64, True)):
        res = h.ld_windows(size, snp_mode=snp)
        exp = restate(c1, c2, pos, off, size, snp)
        assert_restated(res, exp, f"{size} {snp}")
        assert snp or exp["empty"].sum() > 10


@pytest.mark.gpu
def test_ecb_subset_vcf_vs_restatement_and_scikit_allel():
    import twoDSFS_class as K
    from test_gpu_wcfst import panel_codes
    vcf, pm = os.path.join(GOLDEN, "ecb_subset.vcf.gz"), os.path.join(GOLDEN, "ecb_subset.popmap.txt")
    inst = K.LikelihoodInference_jointSFS(vcf, pm)
    P = inst.make_packed_panel()
    c1, c2 = panel_codes(P)
    for size, snp in ((20000, False), (500000, False), (300, True)):
        got = inst.ld_scan_bySNPs(P, size) if snp else inst.ld_scan(P, size)
        eng = inst._eng()
        res = eng.h.fetch_ld_windows(eng.h.candidates(size, snp))
        exp = restate(c1, c2, P.pos, P.off, size, snp)
        assert_restated(res, exp, f"ecb {size}")
        live = ~exp["empty"]
        assert len(got) == int(live.sum())
        for v, k in zip(got.values(), np.flatnonzero(live)):
            assert v["pairs_pop1"] == exp["n_pairs_p1"][k] and v["sites_pop2"] == exp["n_sites_p2"][k]
            for name, col in (("ZnS_pop1", "zns_p1"), ("omega_pop2", "omega_p2")):
                assert (v[name] is None) == bool(np.isnan(exp[col][k])) and (v[name] is None or v[name] == exp[col][k])
            assert (v["omega_pos_pop1"] is None) == (exp["omega_pos_p1"][k] < 0)
        if size == 500000:  # scikit-allel's pairwise r, literally, over the biggest windows
            wins = candidate_windows(P.pos, P.off, size, snp)
            for w, (_, lo, hi, _, _) in enumerate(wins):
                for p, c in ((1, c1), (2, c2)):
                    r2 = skallel_r2(DOSE[c[lo:hi].astype(np.int64)]).astype(np.float64)
                    ok = np.isfinite(r2)
                    assert exp[f"n_pairs_p{p}"][w] == int(ok.sum())
                    if ok.any():
                        assert abs(exp[f"zns_p{p}"][w] - r2[ok].mean()) <= F32_TOL + 2.0 ** -32, (w, p)
        assert any(v["omega_pop1"] is not None for v in got.values())


@pytest.mark.gpu
def test_fixups_count_as_missing_and_filters():
    import twoDSFS_class as K
    from tdsfs_engine import filter_flags
    from test_gpu_wcfst import panel_codes
    vcf, pm = os.path.join(GOLDEN, "ingest_small.vcf.gz"), os.path.join(GOLDEN, "ingest_small.popmap.txt")
    for ctor in ({}, dict(start_position=8, end_position=60)):
        inst = K.LikelihoodInference_jointSFS(vcf, pm, pop1_size=3, pop2_size=3, **ctor)
        P = inst.make_packed_panel()
        assert P.fixups is not None and len(P.fixups) > 0
        c1, c2 = panel_codes(P)   # fix-up calls are code 2 here
        flags = filter_flags(P, ctor.get("start_position"), ctor.get("end_position"), None)
        for size, snp in ((30, False), (4, True)):
            got = inst.ld_scan_bySNPs(P, size) if snp else inst.ld_scan(P, size)
            eng = inst._eng()
            res = eng.h.fetch_ld_windows(eng.h.candidates(size, snp))
            assert_restated(res, restate(c1, c2, P.pos, P.off, size, snp, flags), f"ingest_small {ctor} {size}")
            assert len(got) == int(((res["flags"] & 8) == 0).sum())


@pytest.mark.gpu
def test_integer_limit_one_window_of_identical_rows(T, h):
    """100,000 identical polymorphic rows in one window: sum q = 2^32 n_pairs, about 2.1e19 > 2^64."""
    S = 100000
    rng = np.random.default_rng(4)
    row = rng.integers(0, 3, 40)
    row[:3] = [0, 1, 2]
    codes = np.tile(codes_of(row), (S, 1))
    pos = np.arange(1, S + 1, dtype=np.int32)
    load(h, codes[:, :21], codes[:, 21:], pos, [0, S])
    for res in (h.ld_windows(S), h.ld_windows(S, snp_mode=True)):
        assert len(res["start"]) == 1
        for p in (1, 2):
            assert res[f"n_sites_p{p}"][0] == S and res[f"n_pairs_p{p}"][0] == S * (S - 1) // 2 == 4999950000
            assert res[f"zns_p{p}"][0] == 1.0 and res[f"omega_p{p}"][0] == 1.0 and res[f"omega_pos_p{p}"][0] == 2


@pytest.mark.gpu
@pytest.mark.parametrize("size,snp", [(3000, False), (400, True)])
def test_shards_equal_whole_bitwise(T, size, snp):
    import tdsfs_dist as D
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(79)
    S, ns1, ns2 = 12000, 200, 200
    c1, c2 = ld_rich_codes(rng, S, ns1, ns2)
    pos, off = random_positions(rng, S, 2, 120000)
    plan = D.make_shard_plan(pos, off, 3, W=None if snp else size, N=size if snp else None, tol=0.0)
    assert any(not p.first for pieces in plan for p in pieces), "the plan must split a chromosome"
    h = T.Handle(0)
    try:
        h.set_panel(ns1, ns2, True)
        G, w1, w2 = pack_codes(c1, c2)
        h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
        whole = h.ld_windows(size, snp_mode=snp)
        assert_restated(whole, restate(c1, c2, pos, off, size, snp), "whole")
        gathered = []
        for pieces in plan:
            a, b = pieces[0].lo, pieces[-1].hi
            Gr, _, _ = pack_codes(c1[a:b], c2[a:b])
            h.load_genotypes(Gr, b - a, w1, w2, ns1, ns2, pos[a:b], D.local_offsets(pieces))
            gathered.append(D.sharded_ld_windows(h, pieces, pos, size, None, snp_mode=snp))
        cat = {k: np.concatenate([p[k] for p in gathered]) for k in whole}
        assert_bitwise(cat, whole, "shards")
    finally:
        h.close()


@pytest.mark.gpu
def test_ld_windows_leave_other_state_alone(T):
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(8)
    S, ns1, ns2, W = 30000, 200, 200, 20000
    c1, c2 = random_codes(rng, S, ns1, ns2)
    pos, off = random_positions(rng, S, 3, 300000)
    G, w1, w2 = pack_codes(c1, c2)

    def run(with_ld):
        h = T.Handle(0)
        try:
            h.set_panel(ns1, ns2, True)
            h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
            h.diversity(7000, fetch=False)
            h.neutrality(900, snp_mode=True, fetch=False)
            h.wcfst(3000, fetch=False)
            keep = h.ld_prune(100, 20, 0.1)
            h.plan(W)
            if with_ld:  # a pending plan, unfetched window-pass results and ld_prune's buffers
                h.ld_windows(5000, fetch=False)
                h.ld_windows(200, snp_mode=True)
            h.background(T.BG_GENOME)
            h.finalize_background()
            res = h.scan(W)
            fused = h.scan_info()[0]
            out = [res, h.fetch_diversity(h.candidates(7000)), h.fetch_neutrality(h.candidates(900, True)),
                   h.fetch_wcfst(h.candidates(3000)), {"keep": keep}]
            h.set_sync(False)
            for _ in range(3):
                h.step_bp(T.BG_GENOME, W)
                if with_ld:  # unfetched scan results and the step graph
                    h.ld_windows(W, fetch=False)
                h.check()
                out.append(h.fetch_results(h.candidates(W)))
            h.set_sync(True)
            out.append({"keep": h.ld_prune(33, 5, 0.5)})
            return fused, out
        finally:
            h.close()

    fa, a = run(True)
    fb, b = run(False)
    assert fa and fb, "the planned scan must stay on the fused path"
    for x, y in zip(a, b):
        assert_bitwise(x, y, "across ld_windows")


@pytest.mark.gpu
def test_error_conventions_and_async(T, h):
    import ctypes as C
    with pytest.raises(T.TdsfsError) as e:
        h.ld_windows(1000)
    assert e.value.code == T.ERR_STATE
    h.set_panel(5, 5, True)
    with pytest.raises(T.TdsfsError) as e:
        h.fetch_ld_windows(10)
    assert e.value.code == T.ERR_STATE
    cnt = np.array([[4, 6, 5, 5]] * 100, dtype=np.uint16)
    pos = np.arange(1, 101, dtype=np.int32) * 50
    h.load_counts(cnt, pos, [0, 100])
    with pytest.raises(T.TdsfsError) as e:
        h.ld_windows(1000)
    assert e.value.code == T.ERR_STATE and "genotype" in str(e.value)
    rng = np.random.default_rng(12)
    S = 20000
    c1, c2 = ld_rich_codes(rng, S, 200, 200)
    pos, off = random_positions(rng, S, 3, 200000)
    load(h, c1, c2, pos, off)
    for size in (0, -3):
        with pytest.raises(T.TdsfsError) as e:
            h.ld_windows(size)
        assert e.value.code == T.ERR_ARG
    n = h.candidates(1000)
    arrs, r = h._alloc_ld_windows(n)
    nw = C.c_int64()
    assert h._L.tdsfs_ld_windows_bp(h._h, C.c_int64(1000), C.byref(r), C.c_int64(n - 1), C.byref(nw)) == T.ERR_ARG
    assert h._L.tdsfs_ld_windows_bp(None, C.c_int64(1000), C.byref(r), C.c_int64(n), C.byref(nw)) == T.ERR_ARG
    assert h._L.tdsfs_fetch_ld_windows(None, C.byref(r), C.c_int64(n), C.byref(nw)) == T.ERR_ARG
    want = {(size, snp): h.ld_windows(size, snp_mode=snp) for size, snp in ((10000, False), (800, True))}
    assert_restated(want[(800, True)], restate(c1, c2, pos, off, 800, True), "sync")
    h.set_sync(False)
    for (size, snp), exp in want.items():
        assert h.ld_windows(size, snp_mode=snp, fetch=False) == len(exp["start"])
        assert_bitwise(h.fetch_ld_windows(h.candidates(size, snp)), exp, f"async {size} {snp}")
    h.set_sync(True)
    # the other passes have their own results
    for fetch in (h.fetch_diversity, h.fetch_neutrality, h.fetch_wcfst):
        with pytest.raises(T.TdsfsError) as e:
            fetch(n)
        assert e.value.code == T.ERR_STATE
    t = h.timings()
    assert t["ld_windows"] > 0 and h.ld_windows_ms() == t["ld_windows"]
