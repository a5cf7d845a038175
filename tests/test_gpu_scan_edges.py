"""The fused scan (k1_fused, the 4-byte records, k3_finish) and the table scorer at the boundaries of their special cases,
against an extended-precision reference of T.

Panels are built from exact per-SNP targets (alt alleles, heterozygotes and missing diploids per population), so every count
is known before the GPU sees it.  Every case asserts which path ran (scan_info = (fused, record bytes)), checks the integer
outputs and the background histograms bit for bit, and T2D / T1D within 1e-9 * max(|T|, 1) of the reference, with exact
0.0 and +inf where the reference gives them.  The largest relative error of each case is printed (pytest -s)."""
import math

import numpy as np
import pytest

import sfs_oracle as O

gpu = pytest.mark.gpu
RTOL = 1e-9
STATS = (("T2D", "n2d", 1), ("T1D_p1", "n1d_p1", 2), ("T1D_p2", "n1d_p2", 4))  # statistic, its N, its None flag

# ------------------------------------------------------------------------------------------- extended-precision reference
LD = np.longdouble
HAVE_LD = np.finfo(LD).nmant >= 63  # x87 80-bit long double: 64-bit significand


def clr_mp(x, b, dps=50):
    """T = 2 sum_bins x ln((x B) / (b N)) over the populated interior bins, in mpmath at `dps` digits."""
    import mpmath
    x, b = [int(v) for v in np.asarray(x).ravel()], [int(v) for v in np.asarray(b).ravel()]
    N, B = sum(x), sum(b)
    with mpmath.workdps(dps):
        return 2 * mpmath.fsum(xi * mpmath.log(mpmath.mpf(xi * B) / (bi * N)) for xi, bi in zip(x, b) if xi)


def clr_ext(x, b):
    """The reference's 2 (logpmf(x; x/N) - logpmf(x; b/B)) of interior count vectors x (window) and b (background), with
    the gammaln terms cancelled (DESIGN.md section 3): T = 2 sum_bins x ln((x B) / (b N)).  x B and b N are exact integers
    below 2^64, so they convert exactly to a 64-bit significand; each term has one rounded division and one logarithm.
    None when N = 0 or B = 0, +inf when a populated bin has b = 0, exactly 0.0 where the reference gives it: a window that
    is its own background, or one populated bin that is also the background's only bin."""
    x = np.asarray(x, dtype=np.int64).ravel()
    b = np.asarray(b, dtype=np.int64).ravel()
    N, B = int(x.sum()), int(b.sum())
    if N == 0 or B == 0:
        return None
    pop = x > 0
    xp, bp = x[pop], b[pop]
    if np.any(bp == 0):
        return math.inf
    if np.array_equal(x, b) or (len(xp) == 1 and int(bp[0]) == B):
        return 0.0
    if not HAVE_LD:
        return float(clr_mp(x, b, 30))
    assert int(xp.max()) * B < 2 ** 63 and int(bp.max()) * N < 2 ** 63
    r = (xp * B).astype(LD) / (bp * N).astype(LD)
    return float(2 * np.sum(xp.astype(LD) * np.log(r)))


def interior(h2, h1a, h1b):
    """Interior vectors of the three likelihoods: 2D without its first and last bin, folded 1D without bins 0 and n."""
    return h2.ravel()[1:-1], O.fold_dense(h1a)[1:-1], O.fold_dense(h1b)[1:-1]


def test_extended_reference_against_mpmath_and_oracle():
    """The extended-precision reference against mpmath at 50 digits, and against the fp64 oracle (clr_dense) to the 1e-9
    tolerance, on a few hundred random spectra up to N = 1e6 (with the None / +inf / 0.0 cases)."""
    rng = np.random.default_rng(2026)
    worst = 0.0
    for it in range(300):
        K = int(rng.integers(1, 400))
        N = int(rng.choice([1, 10, 1000, 50000, 1000000]))
        p = rng.dirichlet(np.full(K, rng.uniform(0.05, 3.0)))
        x = rng.multinomial(N, p)
        b = rng.multinomial(int(rng.integers(N, 20 * N + 2)), 0.7 * p + 0.3 / K) + (rng.random(K) < 0.9)
        b = np.maximum(b, x > 0)  # +inf is checked below
        if it % 10 == 0:
            b = x.copy()
        t = clr_ext(x, b)
        if it % 10 == 0:
            assert t == 0.0
        m = float(clr_mp(x, b))
        bound = 16 * np.finfo(LD).eps * float(np.sum(x * (1 + np.abs(np.log(np.maximum(x, 1) * b.sum() / (np.maximum(b, 1) * x.sum()))))))
        assert abs(t - m) <= bound + 1e-300, (it, t, m, bound)
        worst = max(worst, abs(t - m) / max(abs(m), 1.0))
        v, none = O.clr_dense(x, b)
        assert not none
        assert abs(v - t) <= RTOL * max(abs(t), 1.0), (it, N, v, t)
    assert worst <= 1e-12, worst
    # None, +inf and the single-bin zero
    assert clr_ext([0, 0], [1, 2]) is None and clr_ext([1, 2], [0, 0]) is None
    assert clr_ext([3, 1], [4, 0]) == math.inf
    assert clr_ext([0, 7, 0], [0, 2, 0]) == 0.0
    t = clr_ext([0, 7, 0], [1, 2, 0])
    assert t != 0.0 and abs(t - 14 * math.log(1.5)) <= 1e-15 * t


# ------------------------------------------------------------------------------------------- panels from exact targets
def codes_from_targets(alt, miss, ns, het=None):
    """2-bit codes [S, ns] (0 = 0/0, 1 = 0/1, 3 = 1/1, 2 = missing) with exactly alt alt alleles, het heterozygotes (default
    alt mod 2) and miss missing diploids per row."""
    alt, miss = np.asarray(alt, dtype=np.int64), np.asarray(miss, dtype=np.int64)
    het = alt % 2 if het is None else np.asarray(het, dtype=np.int64)
    hom = (alt - het) // 2
    assert np.all(hom >= 0) and np.all((alt - het) % 2 == 0) and np.all(hom + het + miss <= ns), "targets do not fit"
    i = np.arange(ns)[None, :]
    c = np.zeros((len(alt), ns), dtype=np.uint8)
    c[i < (hom + het + miss)[:, None]] = 2
    c[i < (hom + het)[:, None]] = 1
    c[i < hom[:, None]] = 3
    return c


def make_panel(alt1, miss1, alt2, miss2, ns1, ns2, het1=None, het2=None):
    """(G in B32 layout, w1, w2, cnt[S, 4] = (ref1, alt1, ref2, alt2)) of a panel with exact per-SNP targets."""
    from tdsfs_pack import pack_codes
    alt1, miss1, alt2, miss2 = (np.asarray(v, dtype=np.int64) for v in (alt1, miss1, alt2, miss2))
    S = len(alt1)
    parts = []
    for a in range(0, S, 65536):  # chunks of whole 32-row blocks: their B32 buffers concatenate
        z = slice(a, min(S, a + 65536))
        G, w1, w2 = pack_codes(codes_from_targets(alt1[z], miss1[z], ns1, None if het1 is None else het1[z]),
                               codes_from_targets(alt2[z], miss2[z], ns2, None if het2 is None else het2[z]))
        parts.append(G)
    cnt = np.stack([2 * (ns1 - miss1) - alt1, alt1, 2 * (ns2 - miss2) - alt2, alt2], axis=1)
    return np.concatenate(parts), w1, w2, cnt


def random_targets(rng, S, ns, lo_miss=0, hi_miss=3):
    miss = np.minimum(rng.integers(lo_miss, hi_miss + 1, size=S), ns)
    f = np.exp(rng.uniform(np.log(0.003), 0.0, size=S))
    alt = np.minimum(rng.binomial(2 * (ns - miss), f), 2 * (ns - miss))
    return alt, miss


def test_panel_helper_counts():
    """codes_from_targets + pack_codes decode (oracle's unpacker) to the targets, including odd widths and padding."""
    rng = np.random.default_rng(1)
    for ns1, ns2 in ((31, 33), (5, 64), (100, 1)):
        a1, m1 = random_targets(rng, 100, ns1)
        a2, m2 = random_targets(rng, 100, ns2)
        G, w1, w2, cnt = make_panel(a1, m1, a2, m2, ns1, ns2)
        assert np.array_equal(O.unpack_counts(G, w1, w2, ns1, ns2, 100), cnt)


# ------------------------------------------------------------------------------------------- reference scan
def ref_scan(cnt, pos, off, n1, n2, W=None, N=None, fold=True, bg="genome", bg_chrom=0, pos_lo=-1, pos_hi=-1):
    """Windows the scan emits (fixed-bp W or fixed-SNP N), scored with clr_ext against the background of `bg`:
    'genome', 'per_chrom' or 'chrom' (chromosome bg_chrom), restricted to positions [pos_lo, pos_hi] when both are >= 0.
    Returns (dict of arrays per emitted window, list of background spectra per group)."""
    cnt = np.asarray(cnt, dtype=np.int64)
    pos = np.asarray(pos, dtype=np.int64)
    off = np.asarray(off, dtype=np.int64)
    C = len(off) - 1
    chrom = np.repeat(np.arange(C), np.diff(off))
    in_bg = np.ones(len(cnt), bool)
    if pos_lo >= 0 and pos_hi >= 0:
        in_bg &= (pos >= pos_lo) & (pos <= pos_hi)

    def spectra(mask):
        return O.dense_spectra(cnt[mask], n1, n2, fold)

    if bg == "genome":
        bgs, group = [spectra(in_bg)], [0] * C
    elif bg == "per_chrom":
        bgs, group = [spectra(in_bg & (chrom == c)) for c in range(C)], list(range(C))
    else:
        bgs, group = [spectra(in_bg & (chrom == bg_chrom))], [0] * C
    bgi = [interior(*g) for g in bgs]
    if W is not None:
        wins = [(c, s, s + W - 1, lo, hi) for c, s, lo, hi in O.bp_window_ranges(pos, off, W)]
    else:
        wins = O.snp_window_ranges(pos, off, N)
    rows = []
    for c, s, e, lo, hi in wins:
        h = O.dense_spectra(cnt[lo:hi], n1, n2, fold)
        if N is not None and h[0].sum() == 0:
            continue  # the reference skips a fixed-SNP window whose 2D spectrum sums to 0
        x = interior(*h)
        rows.append((c, s, e, hi - lo) + tuple(int(v.sum()) for v in x) +
                    tuple(clr_ext(xv, bv) for xv, bv in zip(x, bgi[group[c]])))
    names = ("chrom", "start", "end", "snp_count", "n2d", "n1d_p1", "n1d_p2", "T2D", "T1D_p1", "T1D_p2")
    cols = list(zip(*rows)) if rows else [[] for _ in names]
    return {k: list(v) for k, v in zip(names, cols)}, bgs


MAX_ERR = {}


def check_scan(T, res, exp, what):
    """Emitted windows, integer columns and flags exactly; T within RTOL of the reference, exact 0.0 / +inf where it has them."""
    live = (res["flags"] & (T.F_EMPTY | T.F_SKIPPED)) == 0
    assert int(live.sum()) == len(exp["start"]), (what, int(live.sum()), len(exp["start"]))
    for k in ("chrom", "start", "end", "snp_count", "n2d", "n1d_p1", "n1d_p2"):
        assert np.array_equal(res[k][live], np.asarray(exp[k], dtype=res[k].dtype)), (what, k)
    worst = 0.0
    for k, _, bit in STATS:
        got, flags = res[k][live], res["flags"][live]
        for i, e in enumerate(exp[k]):
            if e is None:
                assert flags[i] & bit, (what, k, i)
                continue
            assert not flags[i] & bit, (what, k, i)
            g = float(got[i])
            if e == 0.0 or math.isinf(e):
                assert g == e, (what, k, i, g, e)  # exact: the reference's 0.0 drives its stale-carry quirk
                continue
            err = abs(g - e) / max(abs(e), 1.0)
            assert err <= RTOL, (what, k, i, g, e, err)
            worst = max(worst, err)
    assert np.all(res["flags"][live] & ~np.uint8(7) == 0), what
    MAX_ERR[what] = max(MAX_ERR.get(what, 0.0), worst)
    print(f"[max rel err] {what}: {worst:.3e}")
    return worst


def check_background(h, bgs, what):
    for g, (h2, h1a, h1b) in enumerate(bgs):
        s2, s1a, s1b = h.get_background(g)
        assert np.array_equal(s2.astype(np.int64), h2), (what, g, "2D")
        assert np.array_equal(s1a.astype(np.int64), h1a), (what, g, "1D pop1")
        assert np.array_equal(s1b.astype(np.int64), h1b), (what, g, "1D pop2")


MODES = {"genome": 2, "per_chrom": 1, "chrom": 3}


def planned(h, size, mode, snp=False, bg_chrom=0, lo=-1, hi=-1):
    h.plan(size, snp_mode=snp)
    h.background(MODES[mode], bg_chrom, lo, hi)
    h.finalize_background()
    return h.scan(size, snp_mode=snp)


def unplanned(h, size, mode, snp=False, bg_chrom=0, lo=-1, hi=-1):
    h.background(MODES[mode], bg_chrom, lo, hi)
    h.finalize_background()
    return h.scan(size, snp_mode=snp)


@pytest.fixture(scope="module")
def T():
    import tdsfs_capi
    return tdsfs_capi


@pytest.fixture()
def h(T):
    hd = T.Handle(0)
    yield hd
    hd.close()


def load(h, G, w1, w2, ns1, ns2, pos, off, n1=None, n2=None, fold=True):
    h.set_panel(ns1 if n1 is None else n1, ns2 if n2 is None else n2, fold)
    h.load_genotypes(G, len(pos), w1, w2, ns1, ns2, np.asarray(pos, dtype=np.int32), np.asarray(off, dtype=np.int64))


# ------------------------------------------------------------------------------------------- 1. WCAP and range snapping
WIN_SIZES = (1, 31, 32, 33, 767, 768, 769)


@pytest.fixture(scope="module")
def wcap_panel():
    """32 + 32 samples, about 2 M rows on 3 chromosomes; fixed-bp windows of W = 10000 hold exactly 1, 31, 32, 33, 767, 768
    or 769 SNPs, cycling, with an empty window now and then."""
    rng = np.random.default_rng(768)
    W, ns = 10000, 32
    pos, off = [], [0]
    for c in range(3):
        p, k = [], 0
        while len(p) < 700000:
            m = WIN_SIZES[(k + c) % len(WIN_SIZES)]
            k += 1 + (k % 11 == 5)  # skip a window now and then
            step = (W - 1) // m
            p.extend(1 + (k - 1) * W + np.arange(m) * step + (k % 3))
        pos += p
        off.append(len(pos))
    pos = np.array(pos, dtype=np.int64)
    S = len(pos)
    a1, m1 = random_targets(rng, S, ns)
    a2, m2 = random_targets(rng, S, ns)
    G, w1, w2, cnt = make_panel(a1, m1, a2, m2, ns, ns)
    return G, w1, w2, cnt, pos.astype(np.int32), np.array(off, dtype=np.int64), W


@gpu
@pytest.mark.parametrize("chunked", [False, True])
def test_wcap_windows_and_range_snapping(T, wcap_panel, monkeypatch, chunked):
    """Windows of exactly 1 .. 769 SNPs with every warp of every CTA owning a range (so range targets fall inside 768-SNP
    windows and snap), once with many small upload chunks (launch ends snap back inside windows too).  Fixed-SNP windows of
    767 and 768 SNPs are fused, 769 goes to the table scorer."""
    G, w1, w2, cnt, pos, off, W = wcap_panel
    ns = 32
    if chunked:
        monkeypatch.setenv("TDSFS_UPLOAD_CHUNK_KB", "96")
    h = T.Handle(0)
    try:
        load(h, G, w1, w2, ns, ns, pos, off)
        exp, bgs = ref_scan(cnt, pos, off, ns, ns, W=W, bg="genome")
        counts = set(exp["snp_count"])
        assert set(WIN_SIZES) <= counts
        res = h.run_bp(T.BG_GENOME, W)
        assert h.scan_info() == (True, 4)
        check_background(h, bgs, "wcap genome")
        check_scan(T, res, exp, f"wcap run_bp chunked={chunked}")
        live = (res["flags"] & T.F_EMPTY) == 0
        assert int(res["snp_count"][live].sum()) == len(pos)
        if chunked:
            return
        res = planned(h, W, "per_chrom")
        assert h.scan_info() == (True, 4)
        exp, bgs = ref_scan(cnt, pos, off, ns, ns, W=W, bg="per_chrom")
        check_background(h, bgs, "wcap per_chrom")
        check_scan(T, res, exp, "wcap per_chrom")
        for N, fused in ((767, True), (768, True), (769, False)):
            res = planned(h, N, "genome", snp=True)
            assert h.scan_info()[0] == fused, N
            exp, _ = ref_scan(cnt, pos, off, ns, ns, N=N, bg="genome")
            check_scan(T, res, exp, f"wcap fixed-SNP {N}")
    finally:
        h.close()


# ------------------------------------------------------------------------------------------- 2. hash table and meta fields
@gpu
def test_hash_table_and_meta_fields(T, h):
    """768-SNP windows with 768 distinct 2D bins, with all 768 SNPs in one bin (multiplicity 768 in the 10-bit field), with
    two bins, and with the most distinct folded 1D bins (31 + 31 at n = 32)."""
    ns, W, m = 32, 100000, 768
    cells = [(a, b) for a in range(0, 2 * ns + 1) for b in range(0, 2 * ns + 1) if 0 < a + b <= 2 * ns]
    rng = np.random.default_rng(9)
    pick = rng.choice(len(cells), size=m, replace=False)
    distinct = np.array([cells[i] for i in pick])
    one = np.tile([[7, 12]], (m, 1))
    two = np.array([[3, 60]] * 384 + [[40, 1]] * 384)
    oned = np.stack([np.arange(m) % 31 + 1, (np.arange(m) * 7) % 31 + 33], axis=1)  # folded 1..31 in both populations
    rnd = np.stack([random_targets(rng, m, ns)[0], random_targets(rng, m, ns)[0]], axis=1)
    blocks = [distinct, one, two, oned, rnd]
    alts = np.concatenate(blocks)
    pos = np.concatenate([1 + k * W + np.arange(m) * 100 for k in range(len(blocks))]).astype(np.int32)
    off = np.array([0, len(pos)], dtype=np.int64)
    z = np.zeros(len(pos), dtype=np.int64)
    G, w1, w2, cnt = make_panel(alts[:, 0], z, alts[:, 1], z, ns, ns)
    load(h, G, w1, w2, ns, ns, pos, off)
    for mode in ("genome", "per_chrom"):
        res = planned(h, W, mode)
        assert h.scan_info() == (True, 4)
        exp, bgs = ref_scan(cnt, pos, off, ns, ns, W=W, bg=mode)
        check_background(h, bgs, f"hash {mode}")
        check_scan(T, res, exp, f"hash table {mode}")
        k1, k2, skip, _, _ = O.counts_to_keys(cnt[:m], ns, ns)
        assert len(set(zip(k1.tolist(), k2.tolist()))) == m and res["n2d"][0] == m
        assert res["n1d_p1"][3] == m and res["n1d_p2"][3] == m


# ------------------------------------------------------------------------------------------- 3. corner, PLAIN and H1CAP
@gpu
@pytest.mark.parametrize("ns1,ns2", [(31, 31), (32, 32), (33, 33), (1023, 1023), (1024, 1024), (31, 1024)])
def test_corner_plain_and_h1cap_edges(T, h, ns1, ns2):
    """2D bins with k = 62 .. 65 in each coordinate (the 64 x 64 shared-memory corner), 1D alt counts 2n - 1 and 2n (at
    n = 1024, 2n = 2048 is the first 1D bin not privatised), genome and per-chromosome backgrounds.  (1024, 1024) has
    2049^2 bins, above the shared-memory scorer's 2^22 limit: it is not fused; (1023, 1023) has 2047^2 and is fused."""
    rng = np.random.default_rng(ns1 * 7 + ns2)
    edge1 = [k for k in (0, 1, 2, 62, 63, 64, 65, 2 * ns1 - 1, 2 * ns1) if k <= 2 * ns1]
    edge2 = [k for k in (0, 1, 2, 62, 63, 64, 65, 2 * ns2 - 1, 2 * ns2) if k <= 2 * ns2]
    grid = np.array([(a, b) for a in edge1 for b in edge2 for _ in range(3)])
    S0 = 1500
    r1, m1 = random_targets(rng, S0, ns1)
    r2, m2 = random_targets(rng, S0, ns2)
    a1 = np.concatenate([grid[:, 0], r1, grid[:, 0]])
    a2 = np.concatenate([grid[:, 1], r2, grid[:, 1][::-1]])
    miss1 = np.concatenate([np.zeros(len(grid), np.int64), m1, np.zeros(len(grid), np.int64)])
    miss2 = np.concatenate([np.zeros(len(grid), np.int64), m2, np.zeros(len(grid), np.int64)])
    S = len(a1)
    G, w1, w2, cnt = make_panel(a1, miss1, a2, miss2, ns1, ns2)
    pos = (np.arange(S) * 37 + 5).astype(np.int32)
    cut = S // 2
    pos[cut:] -= pos[cut] - 3
    off = np.array([0, cut, S], dtype=np.int64)
    W = 20000
    load(h, G, w1, w2, ns1, ns2, pos, off)
    fused = (2 * ns1 + 1) * (2 * ns2 + 1) < (1 << 22) - 1  # score_small_ok: the 10-bit multiplicity beside the bin
    for mode in ("genome", "per_chrom"):
        res = planned(h, W, mode)
        assert h.scan_info() == (fused, 4), (ns1, ns2, h.scan_info())
        exp, bgs = ref_scan(cnt, pos, off, ns1, ns2, W=W, bg=mode)
        check_background(h, bgs, f"corner {ns1},{ns2} {mode}")
        check_scan(T, res, exp, f"corner {ns1},{ns2} {mode}")


# ------------------------------------------------------------------------------------------- 4. the narrow record's d field
def swapped_d_panel(rng, ns, d, S=3000):
    """Random rows plus, in each chromosome, swapped SNPs with d missing diploids in population 1 (alt1 + alt2 > n1 + n2)."""
    a1, m1 = random_targets(rng, S, ns)
    a2, m2 = random_targets(rng, S, ns)
    hot = np.arange(5, S, 97)
    m1[hot] = d
    a1[hot] = 2 * (ns - d) - rng.integers(0, 4, size=len(hot))
    a2[hot] = 2 * ns - rng.integers(0, 3, size=len(hot))
    m2[hot] = 0
    assert np.all(a1[hot] + a2[hot] > 2 * ns)
    G, w1, w2, cnt = make_panel(a1, m1, a2, m2, ns, ns)
    pos = np.concatenate([np.arange(S // 2) * 53 + 1, np.arange(S - S // 2) * 53 + 1]).astype(np.int32)
    return G, w1, w2, cnt, pos, np.array([0, S // 2, S], dtype=np.int64)


@gpu
@pytest.mark.parametrize("ns,md", [(500, 6), (1023, 5)])
def test_narrow_d_field_edge(T, h, ns, md):
    """A swapped SNP with 2^md - 1 missing diploids stays in a 4-byte record; one more falls back to 8-byte records.  Both
    writers (the PLAIN count kernel under a genome background, the generic sink under per-chromosome backgrounds), through
    run_bp and through the step-by-step calls; the results equal the reference either way."""
    W = 40000
    for d, rb in (((1 << md) - 1, 4), (1 << md, 8)):
        G, w1, w2, cnt, pos, off = swapped_d_panel(np.random.default_rng(d + ns), ns, d)
        for mode in ("genome", "per_chrom"):
            exp, bgs = ref_scan(cnt, pos, off, ns, ns, W=W, bg=mode)
            load(h, G, w1, w2, ns, ns, pos, off)
            res = h.run_bp(MODES[mode], W)
            assert h.scan_info() == (True, rb), (d, mode, h.scan_info())
            check_background(h, bgs, f"d={d} {mode}")
            check_scan(T, res, exp, f"narrow d={d} ns={ns} {mode} run_bp")
            load(h, G, w1, w2, ns, ns, pos, off)
            res = planned(h, W, mode)
            assert h.scan_info() == (True, rb), (d, mode, h.scan_info())
            check_scan(T, res, exp, f"narrow d={d} ns={ns} {mode} steps")


# ------------------------------------------------------------------------------------------- 5. declared n vs sample columns
@gpu
@pytest.mark.parametrize("extra,rb", [(1, 4), (70, 8)])
def test_declared_panel_larger_than_samples(T, h, extra, rb):
    """n = ns + 1 keeps narrow records (d = (n - ns) + #missing fits 6 bits), n = ns + 70 does not (d >= 70 > 2^5 - 1 at the
    declared n): the scan equals the reference computed at the declared n, in both writers."""
    ns = 500
    n = ns + extra
    rng = np.random.default_rng(extra)
    S = 4000
    a1, m1 = random_targets(rng, S, ns, 0, 2)
    a2, m2 = random_targets(rng, S, ns, 0, 2)
    hot = np.arange(3, S, 41)
    a1[hot], a2[hot] = 2 * (ns - m1[hot]) - 1, 2 * (ns - m2[hot])  # swapped at the declared n
    G, w1, w2, cnt = make_panel(a1, m1, a2, m2, ns, ns)
    pos = (np.arange(S) * 31 + 1).astype(np.int32)
    off = np.array([0, 1500, S], dtype=np.int64)
    pos[1500:] = (np.arange(S - 1500) * 31 + 1)
    load(h, G, w1, w2, ns, ns, pos, off, n1=n, n2=n)
    for mode in ("genome", "per_chrom"):
        exp, bgs = ref_scan(cnt, pos, off, n, n, W=20000, bg=mode)
        res = h.run_bp(MODES[mode], 20000)
        assert h.scan_info() == (True, rb), h.scan_info()
        check_background(h, bgs, f"n=ns+{extra} {mode}")
        check_scan(T, res, exp, f"n=ns+{extra} {mode}")
        res = planned(h, 300, mode, snp=True)
        assert h.scan_info() == (True, rb)
        exp, _ = ref_scan(cnt, pos, off, n, n, N=300, bg=mode)
        check_scan(T, res, exp, f"n=ns+{extra} {mode} fixed-SNP")


@gpu
@pytest.mark.parametrize("ns", [40, 2100])
def test_declared_panel_smaller_than_samples(T, h, ns):
    """More sample columns than the declared n: a count above 2n is a range error, from the ring kernel (40 samples) and from
    k1_genotypes_wide (2100 + 2100 samples, rows above 4096 samples); with every count within 2n the scan runs normally."""
    n = ns - 5
    rng = np.random.default_rng(ns)
    S = 2000
    a1 = rng.integers(0, 2 * n + 1, size=S)
    a2 = rng.integers(0, 2 * n + 1, size=S)
    z = np.zeros(S, dtype=np.int64)
    m = np.full(S, 5, dtype=np.int64)  # 5 missing diploids: every count stays within 2n
    pos = (np.arange(S) * 17 + 1).astype(np.int32)
    off = np.array([0, S], dtype=np.int64)
    G, w1, w2, cnt = make_panel(a1, m, a2, m, ns, ns)
    load(h, G, w1, w2, ns, ns, pos, off, n1=n, n2=n)
    exp, bgs = ref_scan(cnt, pos, off, n, n, W=5000, bg="genome")
    res = h.run_bp(T.BG_GENOME, 5000)
    assert h.scan_info() == (2 * ns <= 4096, 8)  # rows above 4096 samples: k1_genotypes_wide, no window sums
    check_background(h, bgs, f"ns>n {ns}")
    check_scan(T, res, exp, f"ns>n within range {ns}")
    bad_a1 = a1.copy()
    bad_a1[S // 2] = 2 * n + 1
    G, w1, w2, _ = make_panel(bad_a1, z, a2, z, ns, ns)
    load(h, G, w1, w2, ns, ns, pos, off, n1=n, n2=n)
    with pytest.raises(T.TdsfsError) as e:
        h.run_bp(T.BG_GENOME, 5000)
    assert e.value.code == T.ERR_RANGE


# ------------------------------------------------------------------------------------------- 6. unfolded spectra
@gpu
def test_unfolded_fused_path(T, h):
    """fold = False through k1_fused and k3_finish: plan + scan and run_bp, fixed-bp and fixed-SNP windows, genome,
    per-chromosome and single-chromosome backgrounds; the unplanned scan agrees."""
    rng = np.random.default_rng(0)
    ns, S = 40, 30000
    a1, m1 = random_targets(rng, S, ns)
    a2, m2 = random_targets(rng, S, ns)
    G, w1, w2, cnt = make_panel(a1, m1, a2, m2, ns, ns)
    off = np.array([0, 9000, 21000, S], dtype=np.int64)
    pos = np.concatenate([np.sort(rng.choice(np.arange(1, 900000), size=b - a, replace=False))
                          for a, b in zip(off[:-1], off[1:])]).astype(np.int32)
    load(h, G, w1, w2, ns, ns, pos, off, fold=False)
    for mode in ("genome", "per_chrom", "chrom"):
        for size, snp in ((20000, False), (250, True)):
            kw = dict(W=size) if not snp else dict(N=size)
            exp, bgs = ref_scan(cnt, pos, off, ns, ns, fold=False, bg=mode, bg_chrom=1, **kw)
            res = planned(h, size, mode, snp=snp, bg_chrom=1)
            assert h.scan_info()[0]
            check_background(h, bgs, f"unfolded {mode}")
            check_scan(T, res, exp, f"unfolded {mode} {'snp' if snp else 'bp'}")
            plain = unplanned(h, size, mode, snp=snp, bg_chrom=1)
            assert not h.scan_info()[0]
            check_scan(T, plain, exp, f"unfolded {mode} {'snp' if snp else 'bp'} table scorer")
        if mode != "chrom":
            res = h.run_bp(MODES[mode], 20000)
            assert h.scan_info()[0]
            check_scan(T, res, ref_scan(cnt, pos, off, ns, ns, W=20000, fold=False, bg=mode)[0], f"unfolded {mode} run_bp")


# ------------------------------------------------------------------------------------------- 7. position-restricted background
@gpu
def test_position_restricted_background(T, h):
    """bg_pos_lo / bg_pos_hi equal to SNP positions (both bounds inclusive); the window that is exactly the restricted region
    scores exactly 0.0; -1 in either bound means no restriction; fused and unplanned scans agree with the reference."""
    rng = np.random.default_rng(17)
    ns, S, W = 64, 20000, 10000
    a1, m1 = random_targets(rng, S, ns)
    a2, m2 = random_targets(rng, S, ns)
    G, w1, w2, cnt = make_panel(a1, m1, a2, m2, ns, ns)
    off = np.array([0, 12000, S], dtype=np.int64)
    pos = np.concatenate([np.sort(rng.choice(np.arange(1, 400000), size=b - a, replace=False))
                          for a, b in zip(off[:-1], off[1:])]).astype(np.int32)
    k = (pos[:12000] - 1) // W
    rows = np.flatnonzero(k == 7)  # window 7 of chromosome 0
    lo, hi = int(pos[rows[0]]), int(pos[rows[-1]])
    assert np.sum((pos >= lo) & (pos <= hi)) > len(rows)  # chromosome 1 holds rows in the region too
    load(h, G, w1, w2, ns, ns, pos, off)
    for mode, bgc in (("genome", 0), ("chrom", 0), ("per_chrom", 0)):
        for plo, phi in ((lo, hi), (lo, -1), (-1, hi), (int(pos[100]), int(pos[100]))):
            exp, bgs = ref_scan(cnt, pos, off, ns, ns, W=W, bg=mode, bg_chrom=bgc, pos_lo=plo, pos_hi=phi)
            res = planned(h, W, mode, bg_chrom=bgc, lo=plo, hi=phi)
            assert h.scan_info() == (True, 4)
            check_background(h, bgs, f"restricted {mode} {plo},{phi}")
            check_scan(T, res, exp, f"restricted {mode} [{plo}, {phi}]")
            plain = unplanned(h, W, mode, bg_chrom=bgc, lo=plo, hi=phi)
            check_scan(T, plain, exp, f"restricted {mode} [{plo}, {phi}] table scorer")
            if mode == "chrom" and (plo, phi) == (lo, hi):
                i = exp["start"].index(1 + 7 * W)
                live = np.flatnonzero((res["flags"] & T.F_EMPTY) == 0)
                assert exp["chrom"][i] == 0
                for k_, _, _ in STATS:
                    assert exp[k_][i] == 0.0 and res[k_][live[i]] == 0.0, k_


# ------------------------------------------------------------------------------------------- 8. N == B without self-background
@gpu
def test_window_count_equal_to_background_count(T, h):
    """Single-chromosome background (chromosome 0: one window of 300 SNPs).  A window on chromosome 1 with the same SNP count
    and 1D spectra but another 2D spectrum takes the per-bin path (N == B) and must still give the right nonzero T2D (and
    exact 0.0 for its identical 1D spectra); a window on chromosome 2 with all SNPs in one bin is the one-bin case there."""
    rng = np.random.default_rng(3)
    ns, m = 40, 300
    a1 = rng.integers(1, 30, size=m)
    a2 = rng.integers(1, 30, size=m)
    perm = rng.permutation(m)
    while np.array_equal(a2[perm], a2):
        perm = rng.permutation(m)
    c1 = (a1, a2)
    c2 = (a1, a2[perm])  # same 1D spectra, other pairs
    c3 = (np.full(m, a1[0]), np.full(m, a2[0]))
    A1 = np.concatenate([c1[0], c2[0], c3[0]])
    A2 = np.concatenate([c1[1], c2[1], c3[1]])
    z = np.zeros(3 * m, dtype=np.int64)
    G, w1, w2, cnt = make_panel(A1, z, A2, z, ns, ns)
    pos = np.tile(np.arange(m) * 10 + 1, 3).astype(np.int32)
    off = np.array([0, m, 2 * m, 3 * m], dtype=np.int64)
    load(h, G, w1, w2, ns, ns, pos, off)
    W = 100000
    exp, bgs = ref_scan(cnt, pos, off, ns, ns, W=W, bg="chrom", bg_chrom=0)
    assert exp["n2d"] == [m, m, m]
    assert exp["T2D"][0] == 0.0 and exp["T2D"][1] not in (0.0, None) and exp["T2D"][2] not in (0.0, None)
    assert exp["T1D_p1"][1] == 0.0
    for f in (planned, unplanned):
        res = f(h, W, "chrom", bg_chrom=0)
        check_background(h, bgs, "N == B")
        check_scan(T, res, exp, f"N == B {f.__name__}")


# ------------------------------------------------------------------------------------------- 9. positions near 2^31
@gpu
@pytest.mark.parametrize("W", [99991, 2 ** 30 + 7, 2 ** 31 - 1])
def test_positions_near_int32_limit(T, h, W):
    """Positions in [2^31 - 2e6, 2^31 - 1] (2^31 - 1 included), the window ends clipped to 0x7FFFFFFF, the multiply-high
    window id; a chromosome holding positions 0 and 1 (both in window 0)."""
    rng = np.random.default_rng(W % 1000)
    ns = 32
    top = 2 ** 31 - 1
    p0 = np.sort(rng.choice(np.arange(top - 2000000, top), size=20000, replace=False))
    p0[-1] = top
    p1 = np.concatenate([[0, 1], np.sort(rng.choice(np.arange(2, 300000), size=3000, replace=False))])
    p2 = np.sort(rng.choice(np.arange(top - 300000, top + 1), size=5000, replace=False))
    pos = np.concatenate([p0, p1, p2]).astype(np.int64)
    off = np.array([0, len(p0), len(p0) + len(p1), len(pos)], dtype=np.int64)
    S = len(pos)
    a1, m1 = random_targets(rng, S, ns)
    a2, m2 = random_targets(rng, S, ns)
    G, w1, w2, cnt = make_panel(a1, m1, a2, m2, ns, ns)
    pos32 = pos.astype(np.int32)
    assert pos32.max() == top
    load(h, G, w1, w2, ns, ns, pos32, off)
    for mode in ("genome", "per_chrom"):
        exp, bgs = ref_scan(cnt, pos, off, ns, ns, W=W, bg=mode)
        res = planned(h, W, mode)
        assert h.scan_info()[0]
        check_background(h, bgs, f"2^31 W={W} {mode}")
        check_scan(T, res, exp, f"2^31 W={W} {mode}")
        plain = unplanned(h, W, mode)
        check_scan(T, plain, exp, f"2^31 W={W} {mode} table scorer")
    res = h.run_bp(T.BG_GENOME, W)
    check_scan(T, res, ref_scan(cnt, pos, off, ns, ns, W=W, bg="genome")[0], f"2^31 W={W} run_bp")


# ------------------------------------------------------------------------------------------- 10. large windows at large N
@gpu
def test_large_windows_against_extended_reference(T, h):
    """Windows of 769, about 20 k and about 500 k SNPs (the CTA path of k3_finish), against the extended-precision reference."""
    rng = np.random.default_rng(500)
    ns = 64
    sizes = [769, 20000, 500000, 3, 769]
    W = 1000000
    pos = np.concatenate([1 + k * W + np.sort(rng.choice(np.arange(W), size=m, replace=False)) for k, m in enumerate(sizes)])
    S = len(pos)
    a1, m1 = random_targets(rng, S, ns)
    a2, m2 = random_targets(rng, S, ns)
    G, w1, w2, cnt = make_panel(a1, m1, a2, m2, ns, ns)
    off = np.array([0, S], dtype=np.int64)
    load(h, G, w1, w2, ns, ns, pos.astype(np.int32), off)
    for mode in ("genome", "per_chrom"):
        exp, bgs = ref_scan(cnt, pos, off, ns, ns, W=W, bg=mode)
        assert exp["snp_count"] == sizes
        res = planned(h, W, mode)
        assert h.scan_info() == (True, 4)
        check_background(h, bgs, f"large {mode}")
        check_scan(T, res, exp, f"large windows {mode}")
        res = unplanned(h, W, mode)
        check_scan(T, res, exp, f"large windows {mode} table scorer")
