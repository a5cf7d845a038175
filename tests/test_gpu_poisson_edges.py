"""The legacy Poisson window scan (tdsfs_set_poisson_background + tdsfs_scan_poisson_bp, twoDSFS.calculate_p_window) on
every scorer path, and tdsfs_poisson_score (twoDSFS.calculate_p), against an mpmath reference.

The score of a window (scripts/twoDSFS.py:336-374, the oracle's poisson_window_score): x is the window's unfolded 2D
spectrum over every bin but (0, 0), the corner included; total = sum x, S_w = total + bins / total, pc = 1 / total, and
    P = sum over the bins with q != 0 of  int(x + pc) ln(S_w q) - S_w q - lgamma(int(x + pc) + 1),   P = 0 when total = 0.
Paths: k3_score_small with one warp per window (windows of at most 768 rows), with two and four warps per window (panels
whose tables leave no room for eight groups in 200 KB), and k3_score_large (windows above 768 rows, and every window of a
panel with (2n1+1)(2n2+1) >= 2^22 - 1).  Rows that fail the spectrum filter or are monomorphic are rows of a window but not
sites: windows of any size can have total 0 or 1.  Every case checks every window: n2d and snp_count exactly, flags 0 or
F_EMPTY, T2D within RTOL * max(|P|, 1) of the reference and exactly 0.0 where P = 0.  The largest relative error of each
case is printed (pytest -s)."""
import math

import numpy as np
import pytest

import sfs_oracle as O
from helpers import GOLDEN, RTOL, close, load_chr1_arrays, load_chr1_dict, rows_to_dict
from test_gpu_scan_edges import make_panel

gpu = pytest.mark.gpu
HASH_SLOTS, WCAP, SCORE_WARPS = 1024, 768, 8


# ------------------------------------------------------------------------------------------- references
class QStats:
    """A background q with the sums poisson_mp needs over its non-zero bins, computed once per panel."""

    def __init__(self, q):
        self.q = np.ascontiguousarray(q, dtype=np.float64).ravel()
        self.vals, self.cnts = np.unique(self.q[self.q != 0], return_counts=True)


def poisson_mp(x, q, dps=40):
    """P in mpmath at `dps` digits.  Every bin with q != 0 contributes k ln(S_w q) - S_w q - loggamma(k + 1), k = int(x + pc)
    (S_w and pc exact).  The populated bins are summed one by one; the empty ones (k = 0, or k = 1 when total = 1) depend
    on q alone and are summed once per distinct value of q, which keeps panels of millions of bins fast when q takes few
    values (backgrounds built from integer counts)."""
    import mpmath
    qs = q if isinstance(q, QStats) else QStats(q)
    x = np.asarray(x, dtype=np.int64).ravel()
    assert x.size == qs.q.size
    total = int(x.sum())
    if total == 0:
        return 0.0
    e = 1 if total == 1 else 0
    pop = np.flatnonzero((x > 0) & (qs.q != 0))
    empty = qs.cnts.copy()
    np.subtract.at(empty, np.searchsorted(qs.vals, qs.q[pop]), 1)
    with mpmath.workdps(dps):
        Sw = mpmath.mpf(total) + mpmath.mpf(x.size) / total

        def term(k, qv):
            mu = Sw * mpmath.mpf(qv)
            return (k * mpmath.log(mu) if k else 0) - mu - mpmath.loggamma(k + 1)

        s = mpmath.fsum(term(int(x[i]) + e, float(qs.q[i])) for i in pop.tolist())
        s += mpmath.fsum(int(c) * term(e, v) for v, c in zip(qs.vals.tolist(), empty.tolist()) if c)
        return float(s)


def poisson_np(x, q):
    """P in fp64, vectorised over every bin (scipy's xlogy and gammaln, one math.fsum)."""
    from scipy.special import gammaln, xlogy
    x = np.asarray(x, dtype=np.int64).ravel()
    q = np.asarray(q, dtype=np.float64).ravel()
    total = int(x.sum())
    if total == 0:
        return 0.0
    Sw = total + x.size / total
    k = (x + (1 if total == 1 else 0))[q != 0].astype(np.float64)
    mu = Sw * q[q != 0]
    return math.fsum((xlogy(k, mu) - mu - gammaln(k + 1.0)).tolist())


def logpmf_sum_mp(x, mu, dps=40):
    """tdsfs_poisson_score's definition in mpmath: sum over mu != 0 of poisson.logpmf(x, mu) = xlogy(x, mu) - mu - lgamma(x + 1)."""
    import mpmath
    with mpmath.workdps(dps):
        return float(mpmath.fsum((int(k) * mpmath.log(mpmath.mpf(m)) if k else 0) - mpmath.mpf(m) - mpmath.loggamma(int(k) + 1)
                                 for k, m in zip(np.asarray(x).tolist(), np.asarray(mu, dtype=np.float64).tolist()) if m != 0))


def golden_windows():
    """(case, window key, x, q, normalised background dict, golden P, window dict) for every window of
    tests/golden/poisson_cases.json."""
    import json
    import os
    out = []
    for c in json.load(open(os.path.join(GOLDEN, "poisson_cases.json")))["cases"]:
        n1, n2 = c["n1"], c["n2"]
        R2 = 2 * n2 + 1
        d = rows_to_dict(c["rows"], ("uv", "bv"))
        src = d if c["bg_rows"] is None else rows_to_dict(c["bg_rows"], ("uv", "bv"))
        bgn = O.legacy_normalize_2d_sfs(O.legacy_calculate_2d_sfs(src, "uv", "bv", n1, n2))
        q = np.zeros((2 * n1 + 1) * R2)
        for (i, j), v in bgn.items():
            q[i * R2 + j] = v
        exp = dict((k, p) for k, p, _ in c["windows"])
        for chrom, ws, win in O.walk_bp(d, c["W"]):
            x = np.zeros_like(q, dtype=np.int64)
            for key, info in win.items():
                a1, a2 = info["calls"].get("uv", (0, 0))[1], info["calls"].get("bv", (0, 0))[1]
                if O._passes(key, info, c["start"], c["end"], c["variant_type"]) and (a1, a2) != (0, 0):
                    x[a1 * R2 + a2] += 1
            key = f"{chrom} {ws}-{ws + c['W'] - 1}"
            out.append((c, key, x, q, bgn, exp[key], win))
    return out


def test_references_on_golden_cases():
    """poisson_np equals the oracle within 1e-12; poisson_mp agrees with the oracle, with legacy_calculate_p and with the
    outputs of the unmodified script within RTOL.  The worst error of the oracle against mpmath is printed."""
    worst = 0.0
    for c, key, x, q, bgn, p_gold, win in golden_windows():
        ora = O.poisson_window_score(x, q)
        leg = O.legacy_calculate_p(O.legacy_calculate_2d_sfs(win, "uv", "bv", c["n1"], c["n2"], c["start"], c["end"],
                                                               c["variant_type"]), bgn)
        mp = poisson_mp(x, q)
        assert abs(poisson_np(x, q) - ora) <= 1e-12 * max(abs(ora), 1.0), (key, poisson_np(x, q), ora)
        for v in (ora, leg, p_gold):
            assert close(v, mp), (key, v, mp)
        worst = max(worst, abs(ora - mp) / max(abs(mp), 1.0))
    print(f"[max rel err] oracle vs mpmath, golden windows: {worst:.3e}")


def test_references_on_random_windows():
    """Windows with total 0, 1, 2 and large on small panels, with q random and 20 % zeros, q[0] != 0, populated bins with
    q = 0 and the corner bin populated: poisson_np equals the oracle within 1e-12 and poisson_mp within RTOL; total = 0 is
    exactly 0 in all three."""
    rng = np.random.default_rng(374)
    worst = 0.0
    for n1, n2 in ((8, 6), (5, 9), (18, 14)):
        bins = (2 * n1 + 1) * (2 * n2 + 1)
        for it in range(12):
            q = rng.random(bins) * (rng.random(bins) >= 0.2)
            q[0] = rng.random() + 0.01
            q /= q[1:-1].sum()
            zero = np.flatnonzero(q[1:] == 0) + 1
            for total in (0, 1, 2, 2, 37, 900):
                x = np.bincount(rng.integers(1, bins, size=total), minlength=bins)
                if total and it % 3 == 0:
                    x[-1] += 1  # the corner
                if total and it % 3 == 1 and len(zero):
                    x[rng.choice(zero)] += 1  # a populated bin with q = 0
                ora = O.poisson_window_score(x, q)
                npv, mp = poisson_np(x, q), poisson_mp(x, q)
                if x.sum() == 0:
                    assert ora == 0.0 and npv == 0.0 and mp == 0.0
                    continue
                assert abs(npv - ora) <= 1e-12 * max(abs(ora), 1.0), (n1, n2, int(x.sum()), npv, ora)
                assert close(mp, ora), (n1, n2, int(x.sum()), mp, ora)
                worst = max(worst, abs(ora - mp) / max(abs(mp), 1.0))
    print(f"[max rel err] oracle vs mpmath, random windows: {worst:.3e}")


def score_group_warps(n1, n2):
    """Warps per window of the Poisson scan's shared-memory scorer, as csrc/tdsfs.cu scan() picks them: G = 1, doubled while
    8 / G tables of score_group_smem_words() words overflow 200 KB.  0: the panel is beyond that scorer and every window
    takes k3_score_large."""
    gwords = HASH_SLOTS + (((n1 + 2) // 2 + (n2 + 2) // 2 + 1) & ~1) + SCORE_WARPS * 10 + 2
    bins = (2 * n1 + 1) * (2 * n2 + 1)
    if not (n1 <= 32767 and n2 <= 32767 and bins < (1 << 22) - 1 and gwords * 4 <= 200 * 1024):
        return 0
    G = 1
    while G < SCORE_WARPS and (SCORE_WARPS // G) * gwords * 4 > 200 * 1024:
        G *= 2
    return G


def table_warps(keys, G):
    """The warps of a G-warp group that own an occupied slot of a window's hash table.  k3_score_small puts bin k at slot
    (k * 0x9E3779B1 mod 2^32) >> 22 with linear probing, and thread tg of the group walks slots tg, tg + 32 G, ...; the set
    of occupied slots of a linear-probing table does not depend on the order of insertion."""
    occ = np.zeros(HASH_SLOTS, dtype=bool)
    for k in sorted(set(int(v) for v in keys if v)):
        s = ((k * 0x9E3779B1) & 0xFFFFFFFF) >> 22
        while occ[s]:
            s = (s + 1) & (HASH_SLOTS - 1)
        occ[s] = True
    return set((np.flatnonzero(occ) % (32 * G) // 32).tolist())


def test_scorer_geometry():
    """The host's choice of warps per window, restated, at the panels the GPU cases use."""
    assert [score_group_warps(*n) for n in ((18, 14), (1023, 1023), (1024, 1024), (10600, 8), (10560, 40), (24000, 8),
                                            (32767, 1))] == [1, 1, 0, 2, 2, 4, 4]
    assert table_warps(range(1, 700), 4) == {0, 1, 2, 3} and table_warps([5], 2) in ({0}, {1})


# ------------------------------------------------------------------------------------------- panels of exact windows
def window_rows(rng, n1, n2, m, t, filler, site, zero_bins, hot):
    """(alt1, alt2, flags) of one window of m rows.  t sites (bit0 set, a bin other than (0, 0)) placed as `site` says:
    'rand', 'corner' (2n1, 2n2), 'qzero' (a bin with q = 0) or 'same' (every site in one bin); the other rows are
    monomorphic ('mono'), fail the spectrum filter ('filtered') or alternate ('mixed').  t = None: m random rows with a
    tenth monomorphic, a tenth filtered, a few corner and q = 0 rows, half the sites in a few hot bins (x >= 2).  About a
    fifth of the rows have bit1 clear (not counted in snp_count)."""
    R1, R2 = 2 * n1 + 1, 2 * n2 + 1
    zero_set = set(zero_bins.tolist())

    def rand_bins(k):
        b = rng.integers(1, R1 * R2 - 1, size=k)
        while zero_set and np.isin(b, zero_bins).any():
            bad = np.isin(b, zero_bins)
            b[bad] = rng.integers(1, R1 * R2 - 1, size=int(bad.sum()))
        return b

    if t is None:
        b = rand_bins(m)
        u = rng.random(m)
        b = np.where(u < 0.5, hot[rng.integers(0, len(hot), size=m)], b)
        b[rng.random(m) < 0.03] = R1 * R2 - 1
        if len(zero_bins):
            qz = rng.random(m) < 0.04
            b[qz] = rng.choice(zero_bins, size=int(qz.sum()))
        b[rng.random(m) < 0.1] = 0
        inc = rng.random(m) >= 0.1
    else:
        if site == "corner":
            sb = [R1 * R2 - 1] + list(rand_bins(t - 1))
        elif site == "qzero":
            sb = [int(rng.choice(zero_bins))] + list(rand_bins(t - 1))
        elif site == "same":
            sb = list(rand_bins(1)) * t
        else:
            sb = list(rand_bins(t))
        filt = {"mono": np.zeros(m - t, bool), "filtered": np.ones(m - t, bool),
                "mixed": np.arange(m - t) % 2 == 1}[filler]
        fb = np.where(filt, rand_bins(m - t), 0)
        b = np.concatenate([np.asarray(sb, dtype=np.int64), fb])
        inc = np.concatenate([np.ones(t, bool), ~filt])
        perm = rng.permutation(m)
        b, inc = b[perm], inc[perm]
    flags = inc.astype(np.uint8) | ((rng.random(m) < 0.8).astype(np.uint8) << 1)
    return b // R2, b % R2, flags


WINDOW_KINDS = [(None, "rand")] + [(t, s) for t in (0, 1, 2) for s in ("rand", "corner", "qzero", "same")
                                   if not (t == 0 and s != "rand") and not (t == 1 and s == "same")]


def build_panel(rng, n1, n2, specs, W=10000, n_chrom=2, zero_bins=None):
    """Fixed-bp windows of width W from specs [(m, t, filler, site)], dealt round-robin over n_chrom chromosomes, every
    fifth window of a chromosome left empty.  Returns alt1, alt2, flags, pos, chrom_off."""
    hot = rng.integers(1, (2 * n1 + 1) * (2 * n2 + 1) - 1, size=24)
    zero_bins = np.zeros(0, np.int64) if zero_bins is None else zero_bins
    hot = hot[~np.isin(hot, zero_bins)]
    per = [[] for _ in range(n_chrom)]
    for i, (m, t, filler, site) in enumerate(specs):
        per[i % n_chrom].append(window_rows(rng, n1, n2, m, t, filler, site, zero_bins, hot))
    a1, a2, fl, pos, off = [], [], [], [], [0]
    for c in range(n_chrom):
        k = 0
        for x1, x2, f in per[c]:
            k += 1 + (k % 5 == 3)
            m = len(x1)
            pos.append(1 + (k - 1) * W + np.sort(rng.choice(W, size=m, replace=False)))
            a1.append(x1); a2.append(x2); fl.append(f)
        off.append(sum(len(v) for v in a1))
    return (np.concatenate(a1), np.concatenate(a2), np.concatenate(fl), np.concatenate(pos).astype(np.int32),
            np.array(off, dtype=np.int64))


def integer_background(rng, bins, zero_bins, q0=True):
    """q from an integer histogram (values 1 .. 15, so q takes few distinct values), zero on zero_bins, q[0] != 0 when q0,
    normalised as the reference does (by every bin but the first and the last)."""
    h = rng.integers(1, 16, size=bins).astype(np.float64)
    h[zero_bins] = 0
    if not q0:
        h[0] = 0
    return h / h[1:-1].sum()


def expected_windows(alt1, alt2, flags, pos, off, n2, W):
    """Per emitted window (chrom, start, end, rows, snp_count, bins of its sites), from the oracle's window walk."""
    R2 = 2 * n2 + 1
    key = alt1.astype(np.int64) * R2 + alt2
    site = ((flags & 1) != 0) & (key != 0)
    out = []
    for c, s, lo, hi in O.bp_window_ranges(pos, off, W):
        out.append((c, s, s + W - 1, hi - lo, int(((flags[lo:hi] >> 1) & 1).sum()), key[lo:hi][site[lo:hi]]))
    return out


MAX_ERR = {}


def check_poisson(T, res, exp, qs, what):
    """Every window: emitted windows, flags, n2d and snp_count exactly; T2D within RTOL of poisson_mp, exactly 0.0 where
    it is 0.  Every failing window is listed: (chrom, start, rows, total, got, expected)."""
    bins = qs.q.size
    live = (res["flags"] & T.F_EMPTY) == 0
    assert np.all(res["flags"][~live] == T.F_EMPTY) and np.all(res["snp_count"][~live] == 0), what
    assert int(live.sum()) == len(exp), (what, int(live.sum()), len(exp))
    L = np.flatnonzero(live)
    for j, k in enumerate(("chrom", "start", "end")):
        assert np.array_equal(res[k][L], np.array([e[j] for e in exp], dtype=res[k].dtype)), (what, k)
    assert np.all(res["flags"][L] == 0), what
    worst, bad = 0.0, []
    for i, (c, s, _, rows, nsnp, keys) in zip(L.tolist(), exp):
        x = np.bincount(keys, minlength=bins)
        total = int(x.sum())
        assert res["n2d"][i] == total and res["snp_count"][i] == nsnp, (what, c, s, res["n2d"][i], total, res["snp_count"][i], nsnp)
        p, g = poisson_mp(x, qs), float(res["T2D"][i])
        err = (0.0 if g == 0.0 else math.inf) if p == 0.0 else abs(g - p) / max(abs(p), 1.0)
        if not err <= RTOL:
            bad.append((c, s, rows, total, g, p))
        else:
            worst = max(worst, err)
    MAX_ERR[what] = worst
    print(f"[max rel err] {what}: {worst:.3e}  ({len(exp)} windows)")
    assert not bad, (what, len(bad), bad[:12])


@pytest.fixture(scope="module")
def T():
    import tdsfs_capi
    return tdsfs_capi


def poisson_scan(T, n1, n2, q, W, counts=None, genotypes=None, flags=None, pos=None, off=None):
    h = T.Handle(0)
    try:
        h.set_panel(n1, n2, False)
        if counts is not None:
            h.load_counts(counts, pos, off, flags=flags)
        else:
            G, w1, w2 = genotypes
            h.load_genotypes(G, len(pos), w1, w2, n1, n2, pos, off, flags=flags)
        h.background(T.BG_NONE)
        h.set_poisson_background(q)
        return h.scan_poisson(W)
    finally:
        h.close()


def counts_of(alt1, alt2, n1, n2):
    return np.stack([2 * n1 - alt1, alt1, 2 * n2 - alt2, alt2], axis=1).astype(np.uint16)


# ------------------------------------------------------------------------------------------- 1. sites per window across WCAP
@pytest.fixture(scope="module")
def wcap_sites_panel():
    """18 + 14 diploids.  Fixed-bp windows of 1, 2, 767, 768 and 769 rows; in each size windows with exactly 0, 1 and 2
    sites (the other rows monomorphic, filtered, or both; the sites random, in the corner, in a bin with q = 0, or sharing
    a bin) and windows of random rows.  q[0] != 0, about 40 bins with q = 0."""
    rng = np.random.default_rng(768)
    n1, n2 = 18, 14
    bins = (2 * n1 + 1) * (2 * n2 + 1)
    zero_bins = rng.choice(np.arange(1, bins - 1), size=40, replace=False)
    specs = []
    for m in (1, 2, 767, 768, 769):
        for t, site in WINDOW_KINDS:
            if t is not None and t > m:
                continue
            fillers = ("mono",) if t == m else ("mono", "filtered", "mixed")
            specs += [(m, t, f, site) for f in fillers]
    a1, a2, flags, pos, off = build_panel(rng, n1, n2, specs, zero_bins=zero_bins)
    q = integer_background(rng, bins, zero_bins)
    miss1 = ((rng.random(len(a1)) < 0.2) & (a1 <= 2 * n1 - 2)).astype(np.int64)
    miss2 = ((rng.random(len(a2)) < 0.2) & (a2 <= 2 * n2 - 2)).astype(np.int64)
    G, w1, w2, cnt = make_panel(a1, miss1, a2, miss2, n1, n2)
    return n1, n2, q, (G, w1, w2), cnt.astype(np.uint16), flags, pos, off


@gpu
@pytest.mark.parametrize("entry", ["genotypes", "counts"])
def test_sites_per_window_across_wcap(T, wcap_sites_panel, entry):
    """Windows of 1 .. 769 rows with 0, 1, 2 and many sites, through both entries: the windows of 769 rows are scored by
    k3_score_large, the others by k3_score_small (one warp per window)."""
    n1, n2, q, geno, cnt, flags, pos, off = wcap_sites_panel
    W = 10000
    exp = expected_windows(cnt[:, 1], cnt[:, 3], flags, pos, off, n2, W)
    qs = QStats(q)
    for m in (1, 2, 767, 768, 769):
        got = {len(k) for _, _, _, r, _, k in exp if r == m}
        assert {0, 1, 2} & set(range(m + 1)) <= got, (m, got)
    assert any(r > WCAP and (k == len(qs.q) - 1).any() for _, _, _, r, _, k in exp)  # the corner in a large window
    assert any(r <= WCAP and (k == len(qs.q) - 1).any() for _, _, _, r, _, k in exp)
    assert any((q[k] == 0).any() for _, _, _, r, _, k in exp if r > WCAP) and q[0] != 0
    if entry == "counts":
        res = poisson_scan(T, n1, n2, q, W, counts=cnt, flags=flags, pos=pos, off=off)
    else:
        res = poisson_scan(T, n1, n2, q, W, genotypes=geno, flags=flags, pos=pos, off=off)
    check_poisson(T, res, exp, qs, f"WCAP sites {entry}")


# ------------------------------------------------------------------------------------------- 2. panels at the scorer limits
@gpu
@pytest.mark.parametrize("n1,n2,G", [(1023, 1023, 1), (1024, 1024, 0), (10600, 8, 2), (24000, 8, 4)])
def test_scorer_limit_panels(T, n1, n2, G):
    """Counts entry.  (1023, 1023): 2047^2 bins, the shared-memory scorer at its 2^22 bin limit.  (1024, 1024): beyond it,
    every window, one-row windows included, takes k3_score_large.  (10600, 8) and (24000, 8): two and four warps per window;
    their windows of random rows occupy table slots of every warp of the group (asserted), and every populated bin there
    has q != 0."""
    assert score_group_warps(n1, n2) == G
    rng = np.random.default_rng(n1 + n2)
    bins = (2 * n1 + 1) * (2 * n2 + 1)
    wide = G > 1
    zero_bins = np.zeros(0, np.int64) if wide else rng.choice(np.arange(1, bins - 1), size=200, replace=False)
    specs = [(m, t, f, s) for m, t, f, s in
             [(1, 0, "mono", "rand"), (1, 0, "filtered", "rand"), (1, 1, "mono", "rand"), (1, 1, "mono", "corner"),
              (2, 0, "mixed", "rand"), (2, 1, "mono", "qzero"), (2, 2, "mono", "same"), (2, 2, "mono", "rand"),
              (300, None, "", ""), (768, 0, "mixed", "rand"), (768, 1, "filtered", "rand"), (768, 2, "mono", "corner"),
              (768, None, "", ""), (768, None, "", ""), (769, 0, "mono", "rand"), (769, 0, "filtered", "rand"),
              (769, 1, "mixed", "qzero"), (769, 1, "mono", "corner"), (769, 2, "mixed", "rand"), (769, None, "", ""),
              (2000, None, "", ""), (2000, 1, "mixed", "rand")]
             if not (wide and s == "qzero")]
    if wide:
        specs += [(1, 1, "mono", "rand")] * 6 + [(700, None, "", "")] * 4
    a1, a2, flags, pos, off = build_panel(rng, n1, n2, specs, zero_bins=zero_bins)
    q = integer_background(rng, bins, zero_bins)
    qs = QStats(q)
    W = 10000
    exp = expected_windows(a1, a2, flags, pos, off, n2, W)
    if wide:
        many = [k for _, _, _, r, _, k in exp if r <= WCAP and len(k) > 100]
        assert len(many) >= 6 and all(table_warps(k, G) == set(range(G)) for k in many)
        assert all((q[k] != 0).all() for _, _, _, _, _, k in exp)
    res = poisson_scan(T, n1, n2, q, W, counts=counts_of(a1, a2, n1, n2), flags=flags, pos=pos, off=off)
    check_poisson(T, res, exp, qs, f"panel {n1},{n2} G={G}")


# ------------------------------------------------------------------------------------------- 3. the drop-in end to end
@pytest.fixture(scope="module")
def chr1():
    d = load_chr1_dict()
    _, pos, cnt, ann, vocab = load_chr1_arrays()
    bgn = O.legacy_normalize_2d_sfs(O.legacy_calculate_2d_sfs(d, "uv", "bv", 18, 14))
    return d, pos.astype(np.int64), cnt.astype(np.int64), ann, vocab, bgn


@gpu
@pytest.mark.parametrize("W", [20000, 500000])
def test_drop_in_rare_annotation_chr1(chr1, W):
    """twoDSFS.calculate_p_window on the chr1 panel (18 + 14 diploids) with variant_type = 'stop_lost' (4 SNPs), with and
    without a start / end pair that cuts inside a window, against the oracle's legacy_calculate_p_window.  At 500 kb the
    windows hold about 10 k rows each and almost all of them no site: windows above 768 rows with 0 and with 1 site are
    asserted to exist.  At 20 kb every window is scored by k3_score_small."""
    import twoDSFS as L
    d, pos, cnt, ann, vocab, bgn = chr1
    vt = "stop_lost"
    wid = (pos - 1) // W
    rows = np.bincount(wid)
    worst = 0.0
    for start, end in ((None, None), (11902000, 19000000)):
        site = (ann == vocab.index(vt)) & ((cnt[:, 1] != 0) | (cnt[:, 3] != 0))
        if start is not None:
            site &= (pos >= start) & (pos <= end)
        sites = np.bincount(wid[site], minlength=len(rows))
        if W == 500000:
            big = rows > WCAP
            assert np.any(big & (sites == 0)) and np.any(big & (sites == 1)), (start, end)
        got = L.calculate_p_window(d, bgn, W, "uv", "bv", 18, 14, start, end, vt)
        exp = O.legacy_calculate_p_window(d, bgn, W, "uv", "bv", 18, 14, start, end, vt)
        assert list(got) == list(exp)
        bad = []
        for k, e in exp.items():
            g = got[k]
            assert g["snp_count"] == e["snp_count"], (k, g, e)
            p, v = e["p_values"], g["p_values"]
            if p == 0:
                ok = v == 0.0
            else:
                ok = abs(v - p) <= RTOL * max(abs(p), 1.0)
                worst = max(worst, abs(v - p) / max(abs(p), 1.0)) if ok else worst
            if not ok:
                bad.append((k, int(rows[(int(k.split(" ")[1].split("-")[0]) - 1) // W]), v, p))
        assert not bad, (W, start, end, len(bad), bad[:12])
    print(f"[max rel err] drop-in chr1 stop_lost W={W}: {worst:.3e}")


# ------------------------------------------------------------------------------------------- 4. tdsfs_poisson_score
@gpu
def test_poisson_score_kernel(T):
    """k_poisson on arrays of 257 .. 4099 bins (every thread of the CTA works) with x = 0, mu = 0 (skipped), x up to 10^6,
    mu down to 1e-300; twoDSFS.calculate_p on fractional foregrounds (int() truncation, pseudo-counts 1 / total and 1)
    against the oracle; both against mpmath."""
    import twoDSFS as L
    rng = np.random.default_rng(289)
    h = T.Handle(0)
    worst = 0.0
    try:
        specials = [([10 ** 6, 10 ** 6, 999983, 0, 1, 5], [1e6, 2.5, 1e6 + 0.5, 1e-300, 1e-300, 0.0]),
                    ([10 ** 6, 0, 3, 0], [1e-300, 0.0, 1e-300, 7.0])]
        for n in (257, 1000, 4099):
            for sx, smu in specials:
                x = rng.integers(0, 40, size=n)
                mu = rng.uniform(0.05, 60.0, size=n)
                x[rng.random(n) < 0.3] = 0
                mu[rng.random(n) < 0.1] = 0.0
                x[:len(sx)], mu[:len(smu)] = sx, smu
                p = rng.permutation(n)
                x, mu = x[p], mu[p]
                got, exp = h.poisson_score(x, mu), logpmf_sum_mp(x, mu)
                assert close(got, exp), (n, got, exp)
                worst = max(worst, abs(got - exp) / max(abs(exp), 1.0))
        n1, n2 = 18, 14
        keys = [(i, j) for i in range(2 * n1 + 1) for j in range(2 * n2 + 1)]
        for it in range(6):
            b = rng.random(len(keys)) * (rng.random(len(keys)) >= 0.2)
            bg = {k: v / b[1:-1].sum() for k, v in zip(keys, b.tolist()) if it % 2 == 0 or v}  # absent keys: .get -> 0
            if it < 4:
                c = rng.integers(0, 6, size=len(keys)) * (rng.random(len(keys)) < 0.3)
                frac = rng.choice([0.0, 1 / 7, 0.5, 0.999999999, 1e-9], size=len(keys))
                fg = {k: int(ci) + float(f) for k, ci, f in zip(keys, c.tolist(), frac.tolist())}
            else:  # windows of one site and two sites as the reference builds them (pseudo-counts 1 and 1/2)
                win = {"c-1": {"calls": {"uv": (30, 6), "bv": (20, 8)}, "annotation": "A"}}
                if it == 5:
                    win["c-2"] = {"calls": {"uv": (36, 0), "bv": (27, 1)}, "annotation": "A"}
                fg = O.legacy_calculate_2d_sfs(win, "uv", "bv", n1, n2)
            S_w = sum(fg.values())
            xs = [int(v) for v in fg.values()]
            mus = [S_w * bg.get(k, 0) for k in fg]
            exp = logpmf_sum_mp(xs, mus)
            got, ora = L.calculate_p(fg, bg), O.legacy_calculate_p(fg, bg)
            assert close(got, exp) and close(ora, exp), (it, got, ora, exp)
            worst = max(worst, abs(got - exp) / max(abs(exp), 1.0))
    finally:
        h.close()
    print(f"[max rel err] tdsfs_poisson_score: {worst:.3e}")


# ------------------------------------------------------------------------------------------- 5. states
@gpu
def test_poisson_states(T):
    """A folded panel refuses the Poisson scan; a handle holding a Poisson background refuses the likelihood scan and the
    other way round; after a Poisson scan, set_background + scan give the likelihood results of a fresh handle bit for bit.
    The windows hold bins with distinct home slots in the scorer's hash table, so their sums are added in one order."""
    rng = np.random.default_rng(5)
    n1, n2, W = 8, 6, 2000
    R1, R2 = 2 * n1 + 1, 2 * n2 + 1
    a1, a2 = [], []
    for w in range(60):  # 40 rows per window over at most 20 bins with distinct home slots
        seen, bins_ = set(), []
        while len(bins_) < 20:
            k = int(rng.integers(1, R1 * R2 - 1))
            s = ((k * 0x9E3779B1) & 0xFFFFFFFF) >> 22
            if s not in seen:
                seen.add(s)
                bins_.append(k)
        b = rng.choice(bins_, size=40)
        a1.append(b // R2); a2.append(b % R2)
    a1, a2 = np.concatenate(a1), np.concatenate(a2)
    S = len(a1)
    pos = (np.arange(S) // 40 * W + 1 + np.arange(S) % 40 * 37).astype(np.int32)
    off = np.array([0, S // 2, S], dtype=np.int64)
    pos[S // 2:] = pos[:S - S // 2]
    z = np.zeros(S, dtype=np.int64)
    G, w1, w2, cnt = make_panel(a1, z, a2, z, n1, n2)
    q = integer_background(rng, R1 * R2, np.array([5, 40]))
    b2d = rng.uniform(0.5, 20.0, size=R1 * R2)
    b1a, b1b = rng.uniform(0.5, 20.0, size=n1 + 1), rng.uniform(0.5, 20.0, size=n2 + 1)

    def fresh(fold):
        h = T.Handle(0)
        h.set_panel(n1, n2, fold)
        h.load_genotypes(G, S, w1, w2, n1, n2, pos, off)
        h.background(T.BG_NONE)
        return h

    h = fresh(True)
    try:
        h.set_poisson_background(q)
        with pytest.raises(T.TdsfsError) as e:
            h.scan_poisson(W)
        assert e.value.code == T.ERR_STATE
    finally:
        h.close()
    ref = fresh(False)
    h = fresh(False)
    try:
        ref.set_background(b2d, b1a, b1b)
        want = ref.scan(W)
        with pytest.raises(T.TdsfsError) as e:
            h.scan_poisson(W)
        assert e.value.code == T.ERR_STATE
        h.set_poisson_background(q)
        with pytest.raises(T.TdsfsError) as e:
            h.scan(W)
        assert e.value.code == T.ERR_STATE
        flags = np.full(S, 3, dtype=np.uint8)
        check_poisson(T, h.scan_poisson(W), expected_windows(a1, a2, flags, pos, off, n2, W), QStats(q), "states Poisson")
        h.set_background(b2d, b1a, b1b)
        got = h.scan(W)
        live = (want["flags"] & T.F_EMPTY) == 0
        assert live.sum() == 60
        for k, v in want.items():
            a, b = (v, got[k]) if k in ("chrom", "start", "end", "snp_count", "flags") else (v[live], got[k][live])
            assert a.dtype == b.dtype and a.tobytes() == b.tobytes(), k
    finally:
        h.close()
        ref.close()
