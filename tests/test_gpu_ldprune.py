"""LD pruning (tdsfs_ld_prune, LikelihoodInference_jointSFS.ld_prune, tdsfs_pack.subset_panel): a numpy restatement of the
definition in DESIGN.md section 7, checked on the CPU against a literal restatement of scikit-allel's locate_unlinked, then
the GPU keep mask against the restatement, exactly.

Definition: samples of both populations pooled; dosage g = 0, 1, 2 for codes 0, 1, 3, code 2 missing.  r^2 of rows i and j
over the n samples called in both: cov = n P - Sx Sy, vx = n Qx - Sx^2, vy = n Qy - Sy^2 (exact integers), r^2 =
float(cov^2) / float(vx vy), undefined when vx vy = 0.  Per chromosome (c0 its first row), rows i < j are tested iff
j - c0 < floor((i - c0) / step) step + size; row j is kept iff no kept row i < j tested with j has r^2 > threshold."""
import gzip
import os

import numpy as np
import pytest

from helpers import GOLDEN

DOSE = np.array([0, 1, -1, 2], dtype=np.int64)  # code -> dosage, -1 = missing


# ------------------------------------------------------------------------------------------- restatement (numpy)
def dosages(codes1, codes2):
    """Pooled dosages [S, ns1 + ns2] (-1 = missing) of 2-bit codes."""
    return np.concatenate([DOSE[np.asarray(codes1, dtype=np.int64)], DOSE[np.asarray(codes2, dtype=np.int64)]], axis=1)


def pair_sums(g, i, j):
    """(n, Sx, Sy, Qx, Qy, P) as int64 arrays for the row pairs (i[k], j[k]) of dosages g."""
    x, y = g[i], g[j]
    both = (x >= 0) & (y >= 0)
    x, y = np.where(both, x, 0), np.where(both, y, 0)
    return both.sum(1), x.sum(1), y.sum(1), (x * x).sum(1), (y * y).sum(1), (x * y).sum(1)


def r2_exact(n, Sx, Sy, Qx, Qy, P):
    """r^2 from the integer sums: uint64 products are exact (cov^2 <= vx vy <= n^4 < 2^64), each converted to fp64 with
    round-to-nearest as float(int) does, one division; NaN where undefined."""
    n, Sx, Sy, Qx, Qy, P = (np.asarray(v, dtype=np.int64) for v in (n, Sx, Sy, Qx, Qy, P))
    cov = n * P - Sx * Sy
    vx, vy = (n * Qx - Sx * Sx).astype(np.uint64), (n * Qy - Sy * Sy).astype(np.uint64)
    den = vx * vy
    num = np.abs(cov).astype(np.uint64) ** 2
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(den == 0, np.nan, num.astype(np.float64) / den.astype(np.float64))


def r2_python(n, Sx, Sy, Qx, Qy, P):
    """The same with Python ints (the definition itself)."""
    n, Sx, Sy, Qx, Qy, P = (int(np.asarray(v).reshape(-1)[0]) for v in (n, Sx, Sy, Qx, Qy, P))
    cov, vx, vy = n * P - Sx * Sy, n * Qx - Sx * Sx, n * Qy - Sy * Sy
    return float("nan") if vx * vy == 0 else float(cov * cov) / float(vx * vy)


def r2_band(codes1, codes2, off, size):
    """band[j, d - 1] = r^2 of rows j - d and j (d = 1 .. size - 1) of one chromosome; NaN where undefined or across a
    chromosome start.  The sums come from fp64 matrix products of 0/1/2 matrices (exact integers far below 2^53)."""
    g = dosages(codes1, codes2)
    S = len(g)
    band = np.full((S, size - 1), np.nan)
    c = (g >= 0).astype(np.float64)
    x = np.where(g >= 0, g, 0).astype(np.float64)
    x2 = x * x
    for a, b in zip(off[:-1], off[1:]):
        for j0 in range(a, b, 256):
            j1 = min(b, j0 + 256)
            i0 = max(a, j0 - size + 1)
            cj, xj, x2j = c[j0:j1], x[j0:j1], x2[j0:j1]
            ci, xi, x2i = c[i0:j1], x[i0:j1], x2[i0:j1]
            # [j, i]: n, Sx (row i), Sy (row j), Qx, Qy, P
            sums = (cj @ ci.T, cj @ xi.T, xj @ ci.T, cj @ x2i.T, x2j @ ci.T, xj @ xi.T)
            r2 = r2_exact(*(np.rint(m).astype(np.int64) for m in sums))
            jj, ii = np.meshgrid(np.arange(j0, j1), np.arange(i0, j1), indexing="ij")
            d = jj - ii
            m = (d >= 1) & (d < size)
            band[jj[m], d[m] - 1] = r2[m]
    return band


def window_pairs(off, size, step):
    """tested[j, d - 1]: rows j - d and j share a window."""
    S = int(off[-1])
    t = np.zeros((S, size - 1), dtype=bool)
    for a, b in zip(off[:-1], off[1:]):
        j = np.arange(a, b)[:, None]
        i = j - np.arange(1, size)[None, :]
        t[a:b] = (i >= a) & (j - a < (i - a) // step * step + size)
    return t


def greedy(band, off, size, step, threshold):
    """Keep mask from the r^2 band: rows in order, a row is dropped when a kept earlier row tested with it has r^2 >
    threshold."""
    S = int(off[-1])
    kill = window_pairs(off, size, step) & (band > threshold)  # NaN compares False: an undefined pair never prunes
    keep = np.ones(S, dtype=bool)
    for j in np.flatnonzero(kill.any(1)):
        d = np.flatnonzero(kill[j]) + 1
        if keep[j - d].any():
            keep[j] = False
    return keep


def ld_keep(codes1, codes2, off, size, step, threshold):
    off = np.asarray(off, dtype=np.int64)
    return greedy(r2_band(codes1, codes2, off, size), off, size, step, threshold)


# ------------------------------------------------------------------------------------------- scikit-allel, literally
def skallel_corrcoef(x, y):
    """gn_corrcoef_int8 (allel/opt/stats.pyx) in float32: sums over the samples called in both, then float32 moments."""
    both = (x >= 0) & (y >= 0)
    n = int(both.sum())
    f = np.float32
    m0, m1 = f(x[both].sum()), f(y[both].sum())
    v0, v1, cov = f((x[both] ** 2).sum()), f((y[both] ** 2).sum()), f((x[both] * y[both]).sum())
    if n == 0 or v0 == 0 or v1 == 0:
        return f(np.nan)
    with np.errstate(invalid="ignore", divide="ignore"):
        m0 /= f(n); m1 /= f(n); v0 /= f(n); v1 /= f(n); cov /= f(n)
        cov -= m0 * m1
        v0 -= m0 * m0
        v1 -= m1 * m1
        return f(np.float64(cov) / np.sqrt(np.float64(v0 * v1)))


def skallel_locate_unlinked(gn, size, step, threshold):
    """locate_unlinked_int8 (allel/opt/stats.pyx) statement by statement, one block."""
    loc = np.ones(len(gn), dtype=bool)
    threshold = np.float32(threshold)
    overlap = size - step
    last = False
    for window_start in range(0, len(gn), step):
        window_stop = window_start + size
        if window_stop > len(gn):
            window_stop = len(gn)
            last = True
        for i in range(window_start, window_stop):
            if loc[i]:
                ii = i + 1 if window_start == 0 else max(i + 1, window_start + overlap)
                for j in range(ii, window_stop):
                    if loc[j]:
                        r = skallel_corrcoef(gn[i], gn[j])
                        if np.float32(r * r) > threshold:
                            loc[j] = False
        if last:
            break
    return loc


def ld_rich_codes(rng, S, ns1, ns2, miss=0.05, copy=0.6, noise=0.15):
    """Codes where a row is often a noisy copy of one of the 30 rows before it: many pairs in LD, many rows pruned."""
    ns = ns1 + ns2
    f = rng.uniform(0.05, 0.95, S)
    g = (rng.random((S, ns)) < f[:, None]).astype(np.int64) + (rng.random((S, ns)) < f[:, None])
    for s in range(1, S):
        if rng.random() < copy:
            src = s - int(rng.integers(1, min(s, 30) + 1))
            g[s] = np.where(rng.random(ns) < noise, rng.integers(0, 3, ns), g[src])
            if rng.random() < 0.2:
                g[s] = 2 - g[s]
    c = np.array([0, 1, 3])[g].astype(np.uint8)
    c[rng.random((S, ns)) < miss] = 2
    return c[:, :ns1], c[:, ns1:]


def codes_of(dose_rows):
    """Dosage rows (-1 missing) -> codes."""
    return np.array([0, 1, 3, 2])[np.asarray(dose_rows)].astype(np.uint8)


# ------------------------------------------------------------------------------------------- CPU: the restatement itself
def test_r2_terms_equal_python_ints():
    rng = np.random.default_rng(3)
    c1, c2 = ld_rich_codes(rng, 300, 40, 23)
    g = dosages(c1, c2)
    i, j = rng.integers(0, 300, 2000), rng.integers(0, 300, 2000)
    sums = pair_sums(g, i, j)
    got = r2_exact(*sums)
    for k in range(len(i)):
        want = r2_python(*(v[k] for v in sums))
        assert (np.isnan(got[k]) and np.isnan(want)) or got[k] == want
    band = r2_band(c1, c2, np.array([0, 300]), 40)
    jj, dd = np.nonzero(np.isfinite(band))
    assert np.array_equal(band[jj, dd], r2_exact(*pair_sums(g, jj - dd - 1, jj)))


@pytest.mark.parametrize("seed,size,step,threshold", [(1, 10, 3, 0.1037), (2, 25, 7, 0.2913), (3, 8, 8, 0.4471),
                                                      (4, 6, 9, 0.1789), (5, 40, 1, 0.3311)])
def test_restatement_matches_scikit_allel(seed, size, step, threshold):
    rng = np.random.default_rng(seed)
    S = 160
    c1, c2 = ld_rich_codes(rng, S, 9, 7, noise=0.3)
    off = np.array([0, 61, S])
    band = r2_band(c1, c2, off, size)
    t = window_pairs(off, size, step)
    gap = np.abs(band[t & np.isfinite(band)] - threshold)
    assert gap.min() >= 1e-5, "a tested pair is within float32 rounding of the threshold: pick another seed"
    keep = greedy(band, off, size, step, threshold)
    gn = dosages(c1, c2)
    ska = np.concatenate([skallel_locate_unlinked(gn[a:b], size, step, threshold) for a, b in zip(off[:-1], off[1:])])
    assert np.array_equal(keep, ska)
    assert 0 < (~keep).sum() < S - 10


def test_known_cases():
    rng = np.random.default_rng(0)
    A = rng.integers(0, 3, 20)
    M, X = np.ones(20, np.int64), np.full(20, -1)

    def keep(rows, size=10, step=1, thr=0.1, off=None, ns1=None):
        c = codes_of(rows)
        ns1 = c.shape[1] // 2 if ns1 is None else ns1
        return ld_keep(c[:, :ns1], c[:, ns1:], [0, len(c)] if off is None else off, size, step, thr).tolist()

    # an identical row and the complement 2 - g: r^2 = 1
    assert keep([A, A, 2 - A]) == [True, False, False]
    assert keep([A, 2 - A]) == [True, False] and keep([A, 2 - A], thr=1.0) == [True, True]
    # monomorphic and all-missing rows are never pruned and never prune
    assert keep([A, M, X, A, M, M, X]) == [True, True, True, False, True, True, True]
    assert keep([M, M], thr=0.0) == [True, True] and keep([X, A], thr=0.0) == [True, True]
    # r^2 exactly 0.25: kept at threshold 0.25 (strict), pruned just below
    x, y = [0, 1, 1, 2], [0, 1, 2, 1]
    assert r2_python(*pair_sums(np.array([x, y]), [0], [1])) == 0.25
    assert keep([x, y], thr=0.25) == [True, True] and keep([x, y], thr=0.2499) == [True, False]
    # A ~ B, B ~ C, A !~ C at 0.5: B is pruned, and a pruned row prunes nothing, so C is kept
    a, b, c = [1, 2, 0, 1, 1, 0], [1, 1, 2, 2, 1, 2], [1, 0, 1, 2, 0, 1]
    assert keep([a, b, c], thr=0.5) == [True, False, True]
    # step > size: rows between windows are never tested
    rows = [A] * 13
    assert keep(rows, size=3, step=5) == [True, False, False, True, True, True, False, False, True, True, True, False, False]
    # windows restart at each chromosome (starts not aligned to the step)
    # (windows [0, 4), [3, 7), [6, 7) and [7, 11), [10, 12): rows 4 and 11 share a window only with pruned rows)
    assert keep([A] * 12, size=4, step=3, off=[0, 7, 12]) == [True, False, False, False, True, False, False,
                                                              True, False, False, False, True]
    # padding samples (the 27 unused bits of population 1's pair) would change r^2 if they counted as 0/0 calls
    x, y = [2, 2, 0, 0, 1], [2, 0, 2, 0, 1]
    r_true = r2_python(*pair_sums(np.array([x, y]), [0], [1]))
    r_pad = r2_python(*pair_sums(np.array([x + [0] * 27, y + [0] * 27]), [0], [1]))
    thr = (r_true + r_pad) / 2
    assert r_pad > thr > r_true
    assert keep([x, y], thr=thr, ns1=5) == [True, True]


# ------------------------------------------------------------------------------------------- CPU: subset_panel
def make_panel(rng, sizes, ns1=7, ns2=5):
    """A hand-built PackedPanel with LD-rich rows, fix-ups and annotations; chromosome c has sizes[c] rows."""
    from tdsfs_pack import _FIX_DT, PackedPanel, pack_codes
    S = int(sum(sizes))
    c1, c2 = ld_rich_codes(rng, S, ns1, ns2)
    P = PackedPanel()
    P.G, P.W1, P.W2 = pack_codes(c1, c2)
    P.ns1, P.ns2, P.n = ns1, ns2, S
    P.off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    P.pos = np.concatenate([np.sort(rng.choice(np.arange(1, 10 * s + 2), size=s, replace=False)) for s in sizes]).astype(np.int64)
    P.chroms = [f"chr{i}" for i in range(len(sizes))]
    P.ann = np.array([f"ann{k % 3}" for k in range(S)], dtype=object)
    fx = np.zeros(6, dtype=_FIX_DT)
    fx["snp"] = sorted(rng.choice(S, size=6, replace=False))
    fx["pop"], fx["dref"], fx["dalt"] = rng.integers(0, 2, 6), 1, 0
    P.fixups = fx
    P.pops = ("uv", "bv")
    P.n_records, P.n_skipped = S + 4, 4
    return P, c1, c2


def test_subset_panel():
    from tdsfs_pack import from_b32, subset_panel, unpack_block
    rng = np.random.default_rng(11)
    P, c1, c2 = make_panel(rng, [9, 5, 12])
    keep = np.ones(P.n, dtype=bool)
    keep[[0, 3, 8]] = False
    keep[9:14] = False           # chromosome 1 loses every row
    P.fixups["snp"] = [1, 2, 5, 10, 16, 20]  # row 10 goes with chromosome 1
    keep[2] = False
    P.last_key_row = 8           # dropped: the nearest kept row before it on chromosome 0 is row 7
    Q = subset_panel(P, keep, (50, 5, 0.2))
    idx = np.flatnonzero(keep)
    assert Q.n == len(idx) and (Q.W1, Q.W2, Q.ns1, Q.ns2, Q.pops) == (P.W1, P.W2, P.ns1, P.ns2, P.pops)
    rows = from_b32(Q.G, Q.n, Q.W1 + Q.W2)
    assert np.array_equal(unpack_block(rows[:, :Q.W1], Q.ns1), c1[idx]) and np.array_equal(unpack_block(rows[:, Q.W1:], Q.ns2), c2[idx])
    assert len(Q.G) == (Q.n + 31) // 32 * 32 * (Q.W1 + Q.W2)
    assert np.array_equal(Q.pos, P.pos[idx]) and list(Q.ann) == list(P.ann[idx])
    assert Q.chroms == ["chr0", "chr2"] and Q.off.tolist() == [0, 5, 5 + 12]
    new = {int(o): n for n, o in enumerate(idx)}
    kept_fx = [f for f in P.fixups if keep[f["snp"]]]
    assert len(Q.fixups) == len(kept_fx) == 4
    assert [(int(f["snp"]), int(f["pop"])) for f in Q.fixups] == [(new[int(f["snp"])], int(f["pop"])) for f in kept_fx]
    assert np.array_equal(Q.counts(), P.counts()[idx])
    assert Q.last_key_row == new[7]
    assert Q.cache_sources == [] and Q.ld_prune == (50, 5, 0.2) and P.ld_prune is None
    assert (Q.n_records, Q.n_skipped) == (P.n_records, P.n_skipped)
    # last_key_row kept: mapped; dropped with no kept row before it on its chromosome: the panel's last kept row
    P.last_key_row = 16
    assert subset_panel(P, keep).last_key_row == new[16]
    P.last_key_row = 10
    assert subset_panel(P, keep).last_key_row == Q.n - 1
    # nothing kept
    E = subset_panel(P, np.zeros(P.n, bool))
    assert E.n == 0 and E.off.tolist() == [0] and E.chroms == [] and E.fixups is None and E.last_key_row == -1
    with pytest.raises(ValueError):
        subset_panel(P, keep[:-1])


def test_pruned_panel_save_load_and_cache(tmp_path):
    import shutil

    import tdsfs_pack as TP
    rng = np.random.default_rng(12)
    P, _, _ = make_panel(rng, [20, 17])
    Q = TP.subset_panel(P, rng.random(P.n) < 0.6, (100, 20, 0.1))
    path = str(tmp_path / "pruned.tdsfspk")
    Q.save(path)
    R = TP.load_panel(path)
    assert R.ld_prune == (100, 20, 0.1) and R.n == Q.n and np.array_equal(np.asarray(R.G), Q.G)
    assert np.array_equal(R.fixups, Q.fixups) and R.last_key_row == Q.last_key_row
    P.save(str(tmp_path / "full.tdsfspk"))
    assert TP.load_panel(str(tmp_path / "full.tdsfspk")).ld_prune is None
    # a pruned panel saved at the VCF's cache path, even stamped with its sources, is never taken for the VCF's cache
    vcf, popmap = str(tmp_path / "x.vcf.gz"), str(tmp_path / "x.popmap.txt")
    shutil.copy(os.path.join(GOLDEN, "ecb_subset.vcf.gz"), vcf)
    shutil.copy(os.path.join(GOLDEN, "ecb_subset.popmap.txt"), popmap)
    full = TP.pack_vcf(vcf, popmap, "uv", "bv")
    pruned = TP.subset_panel(full, np.arange(full.n) % 2 == 0, (10, 1, 0.5))
    cache = vcf + ".uv.bv.tdsfspk"
    pruned.save(cache, sources=(vcf, popmap))
    got = TP.cached_pack_vcf(vcf, popmap, "uv", "bv")
    assert got.n == full.n and got.ld_prune is None and np.array_equal(np.asarray(got.G), np.asarray(full.G))
    assert TP.load_panel(cache).ld_prune is None  # rebuilt in place


def test_ld_prune_rejects_a_data_dict():
    import twoDSFS_class as K
    from helpers import rows_to_dict
    inst = K.LikelihoodInference_jointSFS("x", "y")
    d = rows_to_dict([["c1", 10, [3, 1], [2, 2], "No annotation"]], ("uv", "bv"))
    with pytest.raises(TypeError, match="make_packed_panel"):
        inst.ld_prune(d)


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


def odd_offsets(rng, S):
    """Chromosome starts aligned neither to 32 nor to the usual steps, with one-row chromosomes."""
    cuts = sorted(set([1, 2, 45, 46, 47] + rng.integers(50, S - 1, 4).tolist()))
    return np.array([0] + cuts + [S], dtype=np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("ns1,ns2,S", [
    (500, 500, 1400),    # 32 + 32 words (compile-time instantiation)
    (200, 200, 1800),    # 14 + 14 words (compile-time instantiation)
    (18, 14, 2500),      # the ECB panel's geometry: runtime word count
    (37, 5, 2500),       # runtime, uneven, padding in both populations
    (2100, 40, 700),     # runtime, more word pairs than one staging pass holds
])
def test_keep_equals_restatement(T, h, ns1, ns2, S):
    from tdsfs_pack import pack_codes
    from test_gpu_diversity import random_codes
    rng = np.random.default_rng(ns1 * 7 + ns2)
    half = S // 2
    r1, r2 = random_codes(rng, half, ns1, ns2)
    l1, l2 = ld_rich_codes(rng, S - half, ns1, ns2)
    c1, c2 = np.concatenate([l1, r1]), np.concatenate([l2, r2])
    c1[rng.random(c1.shape) < 0.02] = 2
    off = odd_offsets(rng, S)
    pos = np.concatenate([np.arange(1, b - a + 1) * 10 for a, b in zip(off[:-1], off[1:])]).astype(np.int32)
    # fix-up rows: their calls are code 2 in the matrix, whatever the fix-ups add to the allele counts
    fx = np.zeros(5, dtype=T.FIXUP_DTYPE)
    fx["snp"] = np.sort(rng.choice(S, 5, replace=False))
    fx["pop"], fx["dref"], fx["dalt"] = 0, 1, 0
    c1[fx["snp"], 0] = 2
    G, w1, w2 = pack_codes(c1, c2)
    h.set_panel(max(ns1, 2), max(ns2, 2), True)
    h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off, fixups=fx)
    pruned = 0
    for size in (2, 33, 100, 1024):
        band = r2_band(c1, c2, off, size)
        for step in (1, 5, 20, size, size + 3):
            for thr in (0.0, 0.1, 0.5, 1.0):
                got = h.ld_prune(size, step, thr)
                exp = greedy(band, off, size, step, thr)
                assert np.array_equal(got, exp), (size, step, thr, np.flatnonzero(got != exp)[:10])
                pruned += int((~exp).sum())
    assert pruned > 1000
    assert h.ld_prune_ms() > 0


@pytest.mark.gpu
def test_known_cases_on_the_gpu(T, h):
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(0)
    A = rng.integers(0, 3, 20)
    M, X = np.ones(20, np.int64), np.full(20, -1)
    x, y = [0, 1, 1, 2] + [-1] * 16, [0, 1, 2, 1] + [-1] * 16
    a, b, c = ([1, 2, 0, 1, 1, 0] + [-1] * 14, [1, 1, 2, 2, 1, 2] + [-1] * 14, [1, 0, 1, 2, 0, 1] + [-1] * 14)
    px, py = [2, 2, 0, 0, 1] + [-1] * 15, [2, 0, 2, 0, 1] + [-1] * 15
    rows = [A, A, 2 - A, A, M, X, A, M, X, x, y, a, b, c, px, py] + [A] * 13
    codes = codes_of(rows)
    off = np.array([0, 9, 11, 14, 16, len(rows)])
    c1, c2 = codes[:, :5], codes[:, 5:]
    G, w1, w2 = pack_codes(c1, c2)
    h.set_panel(5, 15, True)
    h.load_genotypes(G, len(rows), w1, w2, 5, 15, np.arange(1, len(rows) + 1, dtype=np.int32), off)
    for size, step, thr in ((10, 1, 0.1), (10, 1, 0.25), (10, 1, 0.2499), (10, 1, 0.5), (3, 5, 0.1), (4, 3, 0.9),
                            (10, 1, 0.0), (10, 1, 1.0)):
        assert np.array_equal(h.ld_prune(size, step, thr), ld_keep(c1, c2, off, size, step, thr)), (size, step, thr)


@pytest.mark.gpu
def test_device_pointer_and_chunked_upload(T, monkeypatch):
    import torch
    from tdsfs_pack import pack_codes
    rng = np.random.default_rng(21)
    S, ns1, ns2 = 6000, 200, 200
    c1, c2 = ld_rich_codes(rng, S, ns1, ns2)
    off = np.array([0, 2500, 2501, S], dtype=np.int64)
    pos = np.concatenate([np.arange(1, b - a + 1) for a, b in zip(off[:-1], off[1:])]).astype(np.int32)
    G, w1, w2 = pack_codes(c1, c2)
    exp = ld_keep(c1, c2, off, 100, 20, 0.2)
    assert (~exp).sum() > 100
    got = []
    for how in ("device", "chunked", "host"):
        if how == "chunked":
            monkeypatch.setenv("TDSFS_UPLOAD_CHUNK_KB", "64")
        else:
            monkeypatch.delenv("TDSFS_UPLOAD_CHUNK_KB", raising=False)
        h = T.Handle(0)
        try:
            h.set_panel(ns1, ns2, True)
            src = torch.from_numpy(G.view(np.int32)).cuda() if how == "device" else G
            h.load_genotypes(src, S, w1, w2, ns1, ns2, pos, off)
            got.append(h.ld_prune(100, 20, 0.2))
        finally:
            h.close()
    for g in got:
        assert np.array_equal(g, exp)


@pytest.mark.gpu
def test_empty_panel(T, h):
    h.set_panel(4, 4, True)
    h.load_genotypes(np.zeros(0, np.uint32), 0, 2, 2, 4, 4, np.zeros(0, np.int32), [0])
    assert h.ld_prune(100, 20, 0.1).shape == (0,)
    h.load_genotypes(np.zeros(0, np.uint32), 0, 2, 2, 4, 4, np.zeros(0, np.int32), [0, 0, 0])
    assert h.ld_prune(2, 1, 0.0).shape == (0,)


def write_vcf_subset(src, dst, kept):
    """Copy of the gzip VCF src with only the records whose (chromosome, position) is in kept."""
    with gzip.open(src, "rt") as f, gzip.open(dst, "wt") as g:
        for line in f:
            if line.startswith("#"):
                g.write(line)
                continue
            cols = line.split("\t", 2)
            if (cols[0], int(cols[1])) in kept:
                g.write(line)


@pytest.mark.gpu
def test_ecb_subset_prune_then_scan_equals_repacked_vcf(tmp_path):
    import shutil

    import twoDSFS_class as K
    from test_gpu_wcfst import panel_codes
    vcf, pm = os.path.join(GOLDEN, "ecb_subset.vcf.gz"), os.path.join(GOLDEN, "ecb_subset.popmap.txt")
    inst = K.LikelihoodInference_jointSFS(vcf, pm)
    P = inst.make_packed_panel()
    c1, c2 = panel_codes(P)
    for size, step, thr in ((50, 5, 0.2), (100, 20, 0.1)):
        Q = inst.ld_prune(P, size, step, thr)
        assert Q.ld_prune == (size, step, thr) and Q.cache_sources == []
        kept = set()  # (chromosome, position) of the kept rows
        for c, name in enumerate(Q.chroms):
            kept.update((name, int(p)) for p in Q.pos[Q.off[c]:Q.off[c + 1]])
        chrom_of = np.repeat(np.arange(len(P.chroms)), np.diff(P.off))
        keep = np.array([(P.chroms[ch], int(p)) in kept for ch, p in zip(chrom_of, P.pos)])
        assert np.array_equal(keep, ld_keep(c1, c2, P.off, size, step, thr))
        assert 0 < Q.n < P.n
        sub_vcf = str(tmp_path / f"pruned_{size}.vcf.gz")
        write_vcf_subset(vcf, sub_vcf, kept)
        shutil.copy(pm, str(tmp_path / "popmap.txt"))
        R = inst.make_packed_panel(sub_vcf, str(tmp_path / "popmap.txt"))
        assert (R.n, R.W1, R.W2, R.ns1, R.ns2, R.chroms, R.last_key_row) == (Q.n, Q.W1, Q.W2, Q.ns1, Q.ns2, Q.chroms, Q.last_key_row)
        assert np.array_equal(np.asarray(R.G), Q.G) and np.array_equal(R.pos, Q.pos) and np.array_equal(R.off, Q.off)
        assert list(R.ann) == list(Q.ann) and np.array_equal(R.counts(), Q.counts())
        for W in (20000, 500000):
            a, b = inst.combined_scan(Q, W), inst.combined_scan(R, W)
            assert a == b and len(a) > 0


@pytest.mark.gpu
def test_prune_leaves_other_results_alone(T):
    from tdsfs_pack import pack_codes
    from test_gpu_diversity import assert_bitwise, random_codes, random_positions
    rng = np.random.default_rng(8)
    S, ns1, ns2, W = 30000, 200, 200, 20000
    c1, c2 = random_codes(rng, S, ns1, ns2)
    pos, off = random_positions(rng, S, 3, 300000)
    G, w1, w2 = pack_codes(c1, c2)

    def run(prune):
        h = T.Handle(0)
        try:
            h.set_panel(ns1, ns2, True)
            h.load_genotypes(G, S, w1, w2, ns1, ns2, pos, off)
            h.diversity(7000, fetch=False)
            h.wcfst(900, snp_mode=True, fetch=False)
            h.plan(W)  # the fused scan sums in a fixed order: bitwise comparable (the table scorer's order is not)
            h.background(T.BG_GENOME)
            h.finalize_background()
            h.scan(W, fetch=False)
            assert h.scan_info()[0]
            if prune:  # unfetched scan and window-pass results
                assert h.ld_prune(100, 20, 0.1).sum() > 0
            out = [h.fetch_diversity(h.candidates(7000)), h.fetch_wcfst(h.candidates(900, True)), h.fetch_results(h.candidates(W))]
            h.plan(W)
            if prune:  # a pending plan
                assert h.ld_prune(33, 5, 0.5).sum() > 0
            h.background(T.BG_GENOME)
            h.finalize_background()
            out.append(h.scan(W))
            assert h.scan_info()[0], "the pending plan must still fuse the next scan"
            return out
        finally:
            h.close()

    for x, y in zip(run(True), run(False)):
        assert_bitwise(x, y, "results across ld_prune")


@pytest.mark.gpu
def test_error_conventions(T, h):
    import ctypes as C
    from tdsfs_pack import pack_codes
    with pytest.raises(T.TdsfsError) as e:
        h.ld_prune(100, 20, 0.1)
    assert e.value.code == T.ERR_STATE
    h.set_panel(5, 5, True)
    cnt = np.array([[4, 6, 5, 5]] * 100, dtype=np.uint16)
    pos = np.arange(1, 101, dtype=np.int32) * 50
    h.load_counts(cnt, pos, [0, 100])
    with pytest.raises(T.TdsfsError) as e:
        h.ld_prune(100, 20, 0.1)
    assert e.value.code == T.ERR_STATE and "genotype" in str(e.value)
    rng = np.random.default_rng(2)
    c1, c2 = ld_rich_codes(rng, 100, 30, 30)
    G, w1, w2 = pack_codes(c1, c2)
    h.load_genotypes(G, 100, w1, w2, 30, 30, pos, [0, 100])
    for size, step, thr in ((1, 1, 0.1), (1025, 1, 0.1), (0, 1, 0.1), (10, 0, 0.1), (10, -2, 0.1), (10, 1, -0.01),
                            (10, 1, 1.01), (10, 1, float("nan")), (10, 1, float("inf"))):
        with pytest.raises(T.TdsfsError) as e:
            h.ld_prune(size, step, thr)
        assert e.value.code == T.ERR_ARG, (size, step, thr)
    n = C.c_int64()
    assert h._L.tdsfs_ld_prune(h._h, C.c_int32(10), C.c_int32(1), C.c_double(0.1), None, C.byref(n)) == T.ERR_ARG
    keep = np.zeros(100, np.uint8)
    assert h._L.tdsfs_ld_prune(h._h, C.c_int32(10), C.c_int32(1), C.c_double(0.1), keep.ctypes.data_as(C.c_void_p), None) == 0
    assert np.array_equal(keep.astype(bool), ld_keep(c1, c2, [0, 100], 10, 1, 0.1))
    assert h.ld_prune(1024, 1, 0.1).shape == (100,)
    t = h.timings()
    assert t["ld_pairs"] > 0 and t["ld_resolve"] > 0 and h.ld_prune_ms() == t["ld_pairs"] + t["ld_resolve"]
