"""The window passes at the integer limits they document (DESIGN.md section 7), against the restatements of
test_gpu_wcfst.py, test_gpu_ldprune.py, test_gpu_diversity.py and test_gpu_neutrality.py and against exact rationals:
Weir and Cockerham's FST at 4000 + 4000 samples, LD pruning at 32767 + 32767 samples (vx vy above 2^63), and the
diversity and neutrality passes on the counts entry at ref, alt = 65535 (2 ref alt and n (n - 1) above 2^32)."""
from fractions import Fraction

import numpy as np
import pytest

from test_gpu_scan_edges import codes_from_targets
from test_gpu_wcfst import assert_restated, code_counts, restate as wc_restate, wc_terms
from test_gpu_ldprune import ld_keep, pair_sums, dosages
from test_gpu_neutrality import assert_matches as neut_matches, restate as neut_restate
from test_gpu_diversity import assert_matches as div_matches, restate as div_restate

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def T():
    import tdsfs_capi
    return tdsfs_capi


@pytest.fixture()
def h(T):
    hd = T.Handle(0)
    yield hd
    hd.close()


def load_codes(h, c1, c2, pos, off, n=None):
    """Load 2-bit codes; n = the declared panel (default: the sample columns)."""
    from tdsfs_pack import pack_codes
    G, w1, w2 = pack_codes(c1, c2)
    h.set_panel(n or c1.shape[1], n or c2.shape[1], True)
    h.load_genotypes(G, len(pos), w1, w2, c1.shape[1], c2.shape[1], np.asarray(pos, dtype=np.int32),
                     np.asarray(off, dtype=np.int64))


# ------------------------------------------------------------------------------------------- Weir and Cockerham at 4000
def wc_rows(ns):
    """(alt, het, missing) per row and population at the extremes of the int64 terms."""
    rows = [
        ((2 * ns, 0, 0), (0, 0, 0)),            # pop 1 all hom-alt, pop 2 all hom-ref: the largest D^2 (N - 1)
        ((0, 0, 0), (2 * ns, 0, 0)),
        ((ns, ns, 0), (ns, ns, 0)),             # all heterozygous
        ((2, 0, ns - 1), (0, 0, ns)),           # one called diploid, in one population only
        ((1, 1, ns - 1), (2 * ns, 0, 0)),       # one called diploid in pop 1 against a full pop 2
        ((2, 0, ns - 1), (1, 1, ns - 2)),       # N = 3
        ((2 * ns - 1, 1, 0), (1, 1, 0)),
        ((ns // 2, ns // 2, 7), (3 * ns // 2, ns // 2, 0)),
    ]
    out = []
    for pop in (0, 1):
        out.append([np.array([r[pop][j] for r in rows]) for j in range(3)])
    return out


def test_wcfst_at_4000_samples(T, h):
    """ns1 = ns2 = 4000: each extreme row alone in a window equals the Python-int restatement bit for bit; the largest
    denominator 4 n1^2 n2^2 (N - 2) is about 8.19e18 < 2^63.  4001 samples: TDSFS_ERR_ARG."""
    ns = 4000
    (a1, h1, m1), (a2, h2, m2) = wc_rows(ns)
    c1, c2 = codes_from_targets(a1, m1, ns, h1), codes_from_targets(a2, m2, ns, h2)
    S = len(a1)
    pos = np.arange(1, S + 1) * 10
    off = [0, S]
    counts = code_counts(c1, c2)
    n1, x1, hh1, n2, x2, hh2 = (int(v[0]) for v in counts)
    assert (n1, x1, n2, x2) == (ns, 2 * ns, ns, 0)
    N = n1 + n2
    assert 4 * n1 * n1 * n2 * n2 * (N - 2) > 8.1e18 and (x1 * n2 - x2 * n1) ** 2 * (N - 1) > 8.1e18
    ab, t = wc_terms(counts)
    assert ab.tolist() == [True, True, True, False, True, True, True, True]
    load_codes(h, c1, c2, pos, off)
    for size, snp in ((1, True), (10, False), (S, True)):
        res = h.wcfst(size, snp_mode=snp)
        assert_restated(res, wc_restate(counts, pos, off, size, snp), f"WC 4000 size {size}")
    c1b = np.concatenate([c1, np.zeros((S, 1), np.uint8)], axis=1)
    load_codes(h, c1b, c2, pos, off)
    with pytest.raises(T.TdsfsError) as e:
        h.wcfst(10)
    assert e.value.code == T.ERR_ARG


# ------------------------------------------------------------------------------------------- LD pruning at 32767 + 32767
def test_ld_prune_at_32767_samples(T, h):
    """Rows of 32767 + 32767 samples (16 KB each) with vx vy >= 2^63: half the samples 0 and half 2, identical, complementary,
    shifted and partly missing copies.  Each pair is its own chromosome (size 2, step 1: only the pair is tested); thresholds
    just below and just above each pair's exact r^2 (fractions.Fraction) decide as the exact value says, and the keep mask
    equals the restatement."""
    ns = 32767
    nt = 2 * ns
    base = np.where(np.arange(nt) < nt // 2, 0, 2)
    rng = np.random.default_rng(32767)
    partners = [base.copy(), 2 - base, np.roll(base, 1), np.roll(base, 1000), np.roll(base, nt // 4),
                np.where(rng.random(nt) < 0.5, base, 1), np.where(np.arange(nt) % 3 == 0, -1, np.roll(base, 77))]
    dose = []
    for p in partners:
        dose += [base, p]
    dose = np.array(dose)
    code = np.array([0, 1, 3, 2])[np.where(dose < 0, 3, dose)].astype(np.uint8)  # dosage -> code, -1 -> missing (2)
    c1, c2 = code[:, :ns], code[:, ns:]
    S = len(dose)
    off = np.arange(0, S + 1, 2)
    pos = np.tile([1, 2], S // 2)
    g = dosages(c1, c2)
    exact, big = [], []
    for i in range(0, S, 2):
        n, Sx, Sy, Qx, Qy, P = (int(v[0]) for v in pair_sums(g, np.array([i]), np.array([i + 1])))
        cov, vx, vy = n * P - Sx * Sy, n * Qx - Sx * Sx, n * Qy - Sy * Sy
        assert vx * vy < 2 ** 64
        big.append(vx * vy >= 2 ** 63)
        exact.append(Fraction(cov * cov, vx * vy))
    assert all(big[:5])  # the last two pairs have missing or half-called samples: smaller products
    assert exact[0] == 1 and exact[1] == 1 and all(0 < r < 1 for r in exact[2:])
    load_codes(h, c1, c2, pos, off, n=5)  # the declared panel only sizes the scan's spectra (2^31 - 1 bins at most)
    for k, r in enumerate(exact):
        for thr, pruned in ((float(r) * (1 - 1e-9), True), (min(1.0, float(r) * (1 + 1e-9)), False)):
            keep = h.ld_prune(2, 1, thr)
            assert np.array_equal(keep, ld_keep(c1, c2, off, 2, 1, thr)), (k, thr)
            assert keep[2 * k + 1] == (not pruned), (k, thr, float(r))


# ------------------------------------------------------------------------------------------- diversity / neutrality at 65535
def frac_rows():
    return np.array([
        [65535, 65535, 65535, 65535],
        [65535, 1, 1, 65535],
        [1, 65535, 65534, 65535],
        [32768, 32767, 65535, 0],
        [65535, 65534, 2, 65535],
        [40000, 65535, 65535, 12345],
        [0, 65535, 65535, 1],
    ], dtype=np.int64)


def test_diversity_and_neutrality_at_uint16_counts(T, h):
    """Counts entry at its uint16 limit: per site pi = 2 ref alt / (n (n - 1)) and dxy = (ref1 alt2 + alt1 ref2) / (n1 n2)
    have numerators and denominators above 2^32.  With each row alone in a window, pi, dxy and theta_pi are the correctly
    rounded quotients of the exact rationals, bit for bit; n_max = 131070 is in the a1 / a2 table."""
    cnt = frac_rows()
    S = len(cnt)
    pos = np.arange(1, S + 1) * 10
    off = [0, S]
    h.set_panel(5, 5, True)
    h.load_counts(cnt.astype(np.uint16), pos, off)
    div = h.diversity(1, snp_mode=True)
    neut = h.neutrality(1, snp_mode=True)
    for i, (r1, a1, r2, a2) in enumerate(cnt.tolist()):
        n1, n2 = r1 + a1, r2 + a2
        pi1, pi2 = float(Fraction(2 * r1 * a1, n1 * (n1 - 1))), float(Fraction(2 * r2 * a2, n2 * (n2 - 1)))
        dxy = float(Fraction(r1 * a2 + a1 * r2, n1 * n2))
        assert (div["pi_p1"][i], div["pi_p2"][i], div["dxy"][i]) == (pi1, pi2, dxy), i
        assert (neut["theta_pi_p1"][i], neut["theta_pi_p2"][i]) == (pi1, pi2), i
        assert (neut["n_max_p1"][i], neut["n_max_p2"][i]) == (n1, n2), i
    assert neut["n_max_p1"][0] == 131070
    for size, snp in ((1, True), (3, True), (1000, False), (25, False)):
        div_matches(h.diversity(size, snp_mode=snp), div_restate(cnt, pos, off, size, snp), f"diversity {size}")
        neut_matches(h.neutrality(size, snp_mode=snp), neut_restate(cnt, pos, off, size, snp), f"neutrality {size}")
