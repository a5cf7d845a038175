"""GPU parity tests proper: the CUDA path, called through the C ABI (ctypes -> libtdsfs.so), against
(a) the reference's shipped golden outputs and (b) the CPU oracle on the same seeded inputs.
Integer work (spectra, window assignment, snp_count) is bit-exact; T2D/T1D within 1e-9 * max(|T|, 1)."""
import os

import numpy as np
import pytest

import sfs_oracle as O
from helpers import GOLDEN, load_chr1_arrays, load_ecb_csv, load_small

pytestmark = pytest.mark.gpu

RTOL = 1e-9


@pytest.fixture(scope="module")
def T():
    import tdsfs_capi
    return tdsfs_capi


@pytest.fixture()
def h(T):
    hd = T.Handle(0)
    yield hd
    hd.close()


def assert_T(got, exp, msg=""):
    got, exp = np.asarray(got, float), np.asarray(exp, float)
    inf = np.isinf(exp)
    assert np.array_equal(np.isinf(got), inf), msg
    assert np.array_equal(got[inf], exp[inf]), msg
    ok = ~inf
    err = np.abs(got[ok] - exp[ok]) / np.maximum(np.abs(exp[ok]), 1.0)
    assert err.size == 0 or err.max() <= RTOL, f"{msg}: max rel err {err.max():.3e}"


def compare_scan(T, res, exp, snp_mode=False):
    """res: C-ABI arrays per candidate; exp: oracle arrays per emitted window."""
    live = (res["flags"] & (T.F_EMPTY | T.F_SKIPPED)) == 0
    assert int(live.sum()) == len(exp["start"]), (int(live.sum()), len(exp["start"]))
    if len(exp["start"]) == 0:
        return
    for k in ("chrom", "start", "end", "snp_count"):
        assert np.array_equal(res[k][live], exp[k]), k
    for a, bit in (("T2D", T.F_T2D_NONE), ("T1D_p1", T.F_T1D_P1_NONE), ("T1D_p2", T.F_T1D_P2_NONE)):
        none = (res["flags"][live] & bit) != 0
        assert np.array_equal(none, exp[a + "_none"].astype(bool)), a
        assert_T(res[a][live][~none], exp[a][~none.astype(bool)], a)


# ------------------------------------------------------------------------------------------- golden KATs (counts entry)
@pytest.fixture(scope="module")
def chr1():
    return load_chr1_arrays()


def test_chr1_background_bit_exact(T, h, chr1):
    chrom, pos, cnt, ann, vocab = chr1
    runs = np.load(os.path.join(GOLDEN, "chr1_ref_runs.npz"))
    h.set_panel(18, 14, True)
    h.load_counts(cnt, pos, [0, len(pos)])
    h.background(T.BG_PER_CHROM)
    s2, s1a, s1b = h.get_background(0)
    assert np.array_equal(s2.astype(np.int64), runs["bg2d"])
    assert np.array_equal(s1a.astype(np.int64), runs["bg1d_uv"])
    assert np.array_equal(s1b.astype(np.int64), runs["bg1d_bv"])


@pytest.mark.parametrize("tag,size,snp", [("20kb", 20000, False), ("500kb", 500000, False), ("500snps", 500, True)])
def test_chr1_shipped_outputs(T, h, chr1, tag, size, snp):
    """data/chr1.pkl.bz2 -> data/ECBstats_*.csv (chromosome 1), the reference's own golden vectors."""
    chrom, pos, cnt, ann, vocab = chr1
    rows = load_ecb_csv(tag)
    h.set_panel(18, 14, True)
    h.load_counts(cnt, pos, [0, len(pos)])
    h.background(T.BG_PER_CHROM)
    h.finalize_background()
    res = h.scan(size, snp_mode=snp)
    live = (res["flags"] & (T.F_EMPTY | T.F_SKIPPED)) == 0
    got = {(int(s), int(e)): i for i, (s, e) in enumerate(zip(res["start"], res["end"])) if live[i]}
    assert len(got) == len(rows)
    for r in rows:
        i = got[(r["window_start"], r["window_end"])]
        assert res["snp_count"][i] == r["snp_count"]
        for a, b, bit in (("T2D", "T2D", T.F_T2D_NONE), ("T1D_p1", "T1D_p1", T.F_T1D_P1_NONE), ("T1D_p2", "T1D_p2", T.F_T1D_P2_NONE)):
            if r[b] is None:
                assert res["flags"][i] & bit, (r, a)
            else:
                assert not (res["flags"][i] & bit)
                assert abs(res[a][i] - r[b]) <= RTOL * max(abs(r[b]), 1.0), (r, a, res[a][i])


def test_chr1_vs_reference_runs_precomputed_float_background(T, h, chr1):
    """scan_precomputed_BG with the NORMALISED whole-chromosome background (class :1970-1983 usage), 100 kb."""
    chrom, pos, cnt, ann, vocab = chr1
    runs = np.load(os.path.join(GOLDEN, "chr1_ref_runs.npz"))
    b2 = runs["bg2d"].astype(np.float64)
    b2n = b2 / b2.ravel()[1:-1].sum()
    f1 = O.fold_dense(runs["bg1d_uv"]).astype(np.float64)
    f2 = O.fold_dense(runs["bg1d_bv"]).astype(np.float64)
    f1n, f2n = f1 / f1[1:-1].sum(), f2 / f2[1:-1].sum()
    h.set_panel(18, 14, True)
    h.load_counts(cnt, pos, [0, len(pos)])
    h.background(T.BG_NONE)
    h.set_background(b2n, f1n, f2n)
    res = h.scan(100000)
    live = (res["flags"] & T.F_EMPTY) == 0
    assert np.array_equal(res["start"][live], runs["p100k_start"])
    assert np.array_equal(res["snp_count"][live], runs["p100k_snp_count"])
    for a, b in (("T2D", "T2D"), ("T1D_p1", "T1D_pop1"), ("T1D_p2", "T1D_pop2")):
        assert not runs[f"p100k_{b}_none"].any()
        assert_T(res[a][live], runs[f"p100k_{b}"], a)


# ------------------------------------------------------------------------------------------- genotype entry vs oracle
def random_panel(rng, S, ns1, ns2, C, L, miss=0.03):
    from tdsfs_pack import pack_codes
    f = np.exp(rng.uniform(np.log(0.002), np.log(0.998), size=S))

    def codes(ns):
        p = np.clip(f + rng.normal(0, 0.05, S) * np.sqrt(f * (1 - f)), 0, 1)[:, None]
        a = (rng.random((S, ns)) < p).astype(np.uint8) + (rng.random((S, ns)) < p).astype(np.uint8)
        c = np.where(a == 2, 3, a).astype(np.uint8)
        c[rng.random((S, ns)) < miss] = 2
        return c

    G, w1, w2 = pack_codes(codes(ns1), codes(ns2))
    sizes = rng.multinomial(S, np.ones(C) / C)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    pos = np.concatenate([np.sort(rng.choice(np.arange(0, L), size=s, replace=False)) for s in sizes]).astype(np.int32)
    return G, w1, w2, pos, off


@pytest.mark.parametrize("n1,n2,S,C,L,W", [
    (18, 14, 20000, 3, 400000, 20000),      # ECB geometry: 2 + 1 words (unaligned rows)
    (5, 5, 30000, 40, 60000, 5000),         # sims geometry: 1 + 1 words, many chromosomes
    (64, 64, 30000, 4, 300000, 10000),      # 4 + 4 words: aligned path
    (200, 200, 40000, 5, 400000, 20000),    # config-4 geometry: 14 + 14 words, hash scorer
    (500, 500, 12000, 2, 200000, 20000),    # config-5 geometry: 32 + 32 words, aligned + rotation
    (100, 37, 9000, 2, 100000, 7000),       # asymmetric
])
@pytest.mark.parametrize("bg", ["per_chrom", "genome"])
def test_genotype_scan_vs_oracle(T, h, n1, n2, S, C, L, W, bg):
    rng = np.random.default_rng(n1 * 1000 + n2 + S)
    G, w1, w2, pos, off = random_panel(rng, S, n1, n2, C, L)
    cnt = O.unpack_counts(G, w1, w2, n1, n2, S)
    h.set_panel(n1, n2, True)
    h.load_genotypes(G, S, w1, w2, n1, n2, pos, off)
    h.background(T.BG_PER_CHROM if bg == "per_chrom" else T.BG_GENOME)
    # spectra bit-exact
    if bg == "genome":
        e2, e1, e1b = O.dense_spectra(cnt, n1, n2)
        s2, s1a, s1b = h.get_background(0)
        assert np.array_equal(s2.astype(np.int64), e2) and np.array_equal(s1a.astype(np.int64), e1) and np.array_equal(s1b.astype(np.int64), e1b)
    else:
        for c in range(C):
            e2, e1, e1b = O.dense_spectra(cnt[off[c]:off[c + 1]], n1, n2)
            s2, s1a, s1b = h.get_background(c)
            assert np.array_equal(s2.astype(np.int64), e2) and np.array_equal(s1a.astype(np.int64), e1) and np.array_equal(s1b.astype(np.int64), e1b)
    h.finalize_background()
    compare_scan(T, h.scan(W), O.scan_arrays(cnt, pos, off, n1, n2, W=W, bg=bg))
    compare_scan(T, h.scan(250, snp_mode=True), O.scan_arrays(cnt, pos, off, n1, n2, N=250, bg=bg), snp_mode=True)


def test_large_windows_and_unfolded(T, h):
    """Windows above the per-warp capacity (768 SNPs) go through the CTA scorer; also fold=False."""
    rng = np.random.default_rng(99)
    n1, n2, S = 30, 40, 50000
    G, w1, w2, pos, off = random_panel(rng, S, n1, n2, 2, 1000000)
    cnt = O.unpack_counts(G, w1, w2, n1, n2, S)
    for fold in (True, False):
        h.set_panel(n1, n2, fold)
        h.load_genotypes(G, S, w1, w2, n1, n2, pos, off)
        h.background(T.BG_PER_CHROM)
        h.finalize_background()
        for W in (100000, 15000):
            res = h.scan(W)
            assert W != 100000 or res["snp_count"].max() > 768
            compare_scan(T, res, O.scan_arrays(cnt, pos, off, n1, n2, W=W, fold=fold))
        compare_scan(T, h.scan(3000, snp_mode=True), O.scan_arrays(cnt, pos, off, n1, n2, N=3000, fold=fold), snp_mode=True)


def test_counts_entry_equals_genotype_entry_and_window_spectra(T, h):
    rng = np.random.default_rng(123)
    n1, n2, S = 25, 9, 8000
    G, w1, w2, pos, off = random_panel(rng, S, n1, n2, 3, 90000)
    cnt = O.unpack_counts(G, w1, w2, n1, n2, S)
    h.set_panel(n1, n2, True)
    h.load_genotypes(G, S, w1, w2, n1, n2, pos, off)
    a = h.run_bp(T.BG_GENOME, 4000)
    h.load_counts(cnt.astype(np.uint16), pos, off)
    b = h.run_bp(T.BG_GENOME, 4000)
    for k in a:
        if a[k].dtype == np.float64:  # fp64 sums run in atomic-arrival order: equal to rounding, not bitwise
            assert np.allclose(a[k], b[k], rtol=1e-11, atol=1e-11, equal_nan=True), k
        else:
            assert np.array_equal(a[k], b[k]), k
    # spectra of single windows (calculate_2d_sfs / calculate_1d_sfs on window_data)
    wins = O.bp_window_ranges(pos, off, 4000)
    live = np.flatnonzero((b["flags"] & T.F_EMPTY) == 0)
    for j in (0, len(wins) // 2, len(wins) - 1):
        c, s, lo, hi = wins[j]
        e2, e1, e1b = O.dense_spectra(cnt[lo:hi], n1, n2)
        s2, s1a, s1b = h.window_spectra(int(live[j]))
        assert np.array_equal(s2.astype(np.int64), e2) and np.array_equal(s1a.astype(np.int64), e1) and np.array_equal(s1b.astype(np.int64), e1b)


def test_filters_flags_and_fixups(T, h):
    """snp_flags (spectrum filter bit0 / count bit1) and half-call fix-ups."""
    rng = np.random.default_rng(7)
    n1, n2, S = 12, 12, 6000
    G, w1, w2, pos, off = random_panel(rng, S, n1, n2, 2, 80000)
    cnt = O.unpack_counts(G, w1, w2, n1, n2, S)
    inc = rng.random(S) < 0.6
    cntb = rng.random(S) < 0.8
    flags = (inc.astype(np.uint8) | (cntb.astype(np.uint8) << 1))
    # fix-ups: samples stored as missing (code 2) contribute extra (dref, dalt)
    fix_rows = np.sort(rng.choice(S, size=200, replace=False))
    fix = np.zeros(len(fix_rows) + 20, dtype=[("snp", "<i8"), ("pop", "<i4"), ("dref", "<i4"), ("dalt", "<i4")])
    cnt_fixed = cnt.copy()
    rows = np.sort(np.concatenate([fix_rows, fix_rows[:20]]))
    for i, r in enumerate(rows):
        pop, dr, da = int(rng.integers(2)), int(rng.integers(0, 2)), int(rng.integers(0, 2))
        # only legal where the row has at least one missing call left to carry it; keep totals within 2n
        if cnt_fixed[r, 2 * pop] + cnt_fixed[r, 2 * pop + 1] + dr + da > 2 * (n1 if pop == 0 else n2):
            dr = da = 0
        fix[i] = (r, pop, dr, da)
        cnt_fixed[r, 2 * pop] += dr
        cnt_fixed[r, 2 * pop + 1] += da
    h.set_panel(n1, n2, True)
    h.load_genotypes(G, S, w1, w2, n1, n2, pos, off, fixups=fix, flags=flags)
    res = h.run_bp(T.BG_PER_CHROM, 5000)
    exp = O.scan_arrays(cnt_fixed, pos, off, n1, n2, W=5000, include=inc)
    # snp_count honours bit1
    exp_count = np.array([cntb[lo:hi].sum() for c, s, lo, hi in O.bp_window_ranges(pos, off, 5000)])
    exp["snp_count"] = exp_count
    compare_scan(T, res, exp)


def test_range_error(T, h):
    """alt count above 2n of the declared panel: the reference raises KeyError (class :433); we raise ERR_RANGE."""
    cnt = np.array([[2, 2, 2, 2], [0, 9, 1, 1]], dtype=np.uint16)
    h.set_panel(2, 2, True)
    h.load_counts(cnt, np.array([5, 9], dtype=np.int32), [0, 2])
    with pytest.raises(T.TdsfsError) as ei:
        h.background(T.BG_GENOME)
    assert ei.value.code == T.ERR_RANGE


def test_empty_and_ragged_inputs(T, h):
    h.set_panel(3, 3, True)
    # empty chromosomes in the middle, single-SNP chromosome, position 0
    cnt = np.array([[5, 1, 4, 2], [3, 3, 6, 0], [2, 4, 1, 5]], dtype=np.uint16)
    pos = np.array([0, 7, 3], dtype=np.int32)
    off = [0, 2, 2, 3, 3]
    h.load_counts(cnt, pos, off)
    res = h.run_bp(T.BG_PER_CHROM, 5)
    exp = O.scan_arrays(cnt, pos, np.array(off), 3, 3, W=5)
    compare_scan(T, res, exp)
    assert h.candidates(10 ** 9) == 2
    # zero SNPs at all
    h.load_counts(np.zeros((0, 4), np.uint16), np.zeros(0, np.int32), [0, 0])
    res = h.run_bp(T.BG_GENOME, 100)
    assert len(res["start"]) == 0


def test_likelihood_kats(T, h):
    """calculate_likelihood_1D on explicit spectra vs the reference's recorded outputs (None / inf / 0.0 / floats)."""
    for lk in load_small()["likelihood"]:
        x = np.array(lk["fg"][1:-1], dtype=np.int64)
        b = np.array(lk["bg"][1:-1], dtype=np.float64)
        val, none = h.likelihood(x, b, float(sum(lk["bg"][1:-1])))
        if lk["cls"] is None:
            assert none
        else:
            assert not none
            assert_T([val], [lk["cls"]], str(lk))


def test_synthetic_generator_statistics(T, h):
    """The on-device synthetic panel (bench input): codes legal, missing rate ~2 %, padding zero, deterministic."""
    import torch
    S, ns1, ns2 = 4096, 200, 200
    w1 = w2 = 14
    g = torch.zeros(((S + 31) // 32 * (w1 + w2) * 32,), dtype=torch.int32, device="cuda")
    h.synth_genotypes(g.data_ptr(), S, 1000, w1, w2, ns1, ns2, 20241004)
    g2 = torch.zeros_like(g)
    h.synth_genotypes(g2.data_ptr(), S, 1000, w1, w2, ns1, ns2, 20241004)
    assert torch.equal(g, g2)
    from tdsfs_pack import from_b32, unpack_block
    Gb = g.cpu().numpy().view(np.uint32)
    G = from_b32(Gb, S, w1 + w2)
    pop1 = unpack_block(G[:, :w1], w1 * 16)
    assert (pop1[:, ns1:] == 0).all()
    miss = (pop1[:, :ns1] == 2).mean()
    assert 0.015 < miss < 0.025
    cnt = O.unpack_counts(Gb, w1, w2, ns1, ns2, S)
    assert cnt.min() >= 0 and (cnt[:, 0] + cnt[:, 1] <= 2 * ns1).all()
    # spectrum is dominated by rare variants (log-uniform ancestral frequency)
    assert (cnt[:, 1] <= 40).mean() > 0.5


def test_panel_beyond_shared_memory_scorer_limits(T, h):
    """(2n1+1)(2n2+1) >= 2^22 bins: every window goes through the CTA scorer with dense global scratch."""
    rng = np.random.default_rng(5)
    n1 = n2 = 1100
    S = 3000
    cnt = np.zeros((S, 4), dtype=np.uint16)
    for p, n in ((0, n1), (1, n2)):
        called = 2 * n - 2 * rng.binomial(n, 0.02, S)
        alt = rng.binomial(called, np.exp(rng.uniform(np.log(0.001), np.log(0.999), S)))
        cnt[:, 2 * p], cnt[:, 2 * p + 1] = called - alt, alt
    pos = np.sort(rng.choice(np.arange(1, 100000), size=S, replace=False)).astype(np.int32)
    off = np.array([0, 1000, S])
    h.set_panel(n1, n2, True)
    h.load_counts(cnt, pos, off)
    res = h.run_bp(T.BG_PER_CHROM, 10000)
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(os.path.dirname(GOLDEN), "..", "oracle")])
    import sfs_oracle_c as OC
    exp = OC.scan(cnt, pos, off, n1, n2, W=10000, bg="per_chrom", nthreads=4)
    compare_scan(T, res, exp)


def test_rows_wider_than_one_ring_stage(T, h):
    """More than 4096 samples per SNP: K1 streams each 32-SNP block in 64-word segments (k1_genotypes_wide)."""
    rng = np.random.default_rng(77)
    n1, n2, S = 2600, 1700, 2500
    G, w1, w2, pos, off = random_panel(rng, S, n1, n2, 2, 200000)
    assert (w1 + w2) * 128 > 32 * 1024
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(os.path.dirname(GOLDEN), "..", "oracle")])
    import sfs_oracle_c as OC
    cnt = OC.decode(G, S, w1, w2, n1, n2, 4)
    h.set_panel(n1, n2, True)
    h.load_genotypes(G, S, w1, w2, n1, n2, pos, off)
    h.background(T.BG_GENOME)
    e2, e1, e1b = O.dense_spectra(cnt, n1, n2)
    s2, s1a, s1b = h.get_background(0)
    assert np.array_equal(s2.astype(np.int64), e2) and np.array_equal(s1a.astype(np.int64), e1) and np.array_equal(s1b.astype(np.int64), e1b)
    res = h.run_bp(T.BG_PER_CHROM, 40000)
    compare_scan(T, res, OC.scan(cnt, pos, off, n1, n2, W=40000, bg="per_chrom", nthreads=4))


def test_peer_exchange_single_rank(T, h):
    """The peer-memory all-reduce with world = 1 (this rank maps only itself): barrier epochs, in-place reduce and the ln
    tables of the one-launch exchange (peer_allreduce_background runs peer_reduce_finalize) all run, and the scan equals the
    plain one.  Two ranks: tests/test_gpu_multi.py."""
    rng = np.random.default_rng(31)
    n1, n2, S = 20, 16, 9000
    G, w1, w2, pos, off = random_panel(rng, S, n1, n2, 3, 120000)
    h.set_panel(n1, n2, True)
    h.load_genotypes(G, S, w1, w2, n1, n2, pos, off)
    plain = h.run_bp(T.BG_GENOME, 6000)
    with pytest.raises(T.TdsfsError) as ei:       # not set up yet
        h.peer_allreduce_background()
    assert ei.value.code == T.ERR_STATE
    h.background(T.BG_GENOME)
    blob = h.peer_export(0, 1)
    assert len(blob) == T.PEER_BLOB_BYTES
    with pytest.raises(T.TdsfsError):             # blob of the wrong rank
        h.peer_import([b"\x01" * T.PEER_BLOB_BYTES])
    blob = h.peer_export(0, 1)
    h.peer_import([blob])
    for _ in range(3):
        h.background(T.BG_GENOME)
        h.peer_allreduce_background()
        s2, s1a, s1b = h.get_background(0)        # the histogram between two exchanges
        h.peer_allreduce_background()             # sum over one rank: unchanged
        h.finalize_background()
        res = h.scan(6000)
    for k in plain:
        if plain[k].dtype == np.float64:
            assert np.allclose(res[k], plain[k], rtol=1e-11, atol=1e-11, equal_nan=True), k
        else:
            assert np.array_equal(res[k], plain[k]), k
    h.background(T.BG_PER_CHROM)                  # several groups: the exchange refuses
    with pytest.raises(T.TdsfsError) as ei:
        h.peer_allreduce_background()
    assert ei.value.code == T.ERR_STATE
    h.peer_close()
    with pytest.raises(T.TdsfsError):
        h.peer_allreduce_background()


def test_capi_error_conventions(T, h):
    """Return codes + tdsfs_last_error(): call-order violations, bad arguments, small result buffers -- never a crash."""
    cnt = np.array([[2, 2, 2, 2], [3, 1, 1, 3], [4, 0, 2, 2]], dtype=np.uint16)
    pos = np.array([5, 9, 40], dtype=np.int32)
    with pytest.raises(T.TdsfsError) as e:   # no panel yet
        h.load_counts(cnt, pos, [0, 3])
    assert e.value.code == 3
    with pytest.raises(T.TdsfsError) as e:
        h.set_panel(0, 5, True)
    assert e.value.code == 1
    h.set_panel(2, 2, True)
    with pytest.raises(T.TdsfsError) as e:   # background before data
        h.background(T.BG_GENOME)
    assert e.value.code == 3
    with pytest.raises(T.TdsfsError) as e:   # chrom_off must end at S
        h.load_counts(cnt, pos, [0, 2])
    assert e.value.code == 1
    h.load_counts(cnt, pos, [0, 3])
    with pytest.raises(T.TdsfsError) as e:   # scan before background
        h.scan(10)
    assert e.value.code == 3
    with pytest.raises(T.TdsfsError) as e:
        h.background(7)
    assert e.value.code == 1
    with pytest.raises(T.TdsfsError) as e:   # background chromosome out of range
        h.background(T.BG_CHROM, bg_chrom=4)
    assert e.value.code == 1
    h.background(T.BG_GENOME)
    with pytest.raises(T.TdsfsError) as e:   # tables not built yet
        h.scan(10)
    assert e.value.code == 3
    h.finalize_background()
    # result capacity too small
    import ctypes as C
    arrs, r = h._alloc_result(1)
    n = C.c_int64()
    rc = h._L.tdsfs_scan_bp(h._h, C.c_int64(10), C.byref(r), C.c_int64(1), C.byref(n))
    assert rc == 1 and b"capacity" in h._L.tdsfs_last_error()
    res = h.scan(10)
    assert len(res["start"]) == 4 and int(((res["flags"] & T.F_EMPTY) == 0).sum()) == 2
    with pytest.raises(T.TdsfsError) as e:   # window index out of range
        h.window_spectra(99)
    assert e.value.code == 1
    # unsorted fix-ups are rejected
    G = np.zeros(32 * 2, dtype=np.uint32)
    fix = np.array([(2, 0, 1, 0), (1, 0, 0, 1)], dtype=T.FIXUP_DTYPE)
    with pytest.raises(T.TdsfsError) as e:
        h.load_genotypes(G, 3, 1, 1, 2, 2, pos, [0, 3], fixups=fix)
    assert e.value.code == 1
    with pytest.raises(T.TdsfsError) as e:   # more sample columns than the words hold
        h.load_genotypes(G, 3, 1, 1, 17, 2, pos, [0, 3])
    assert e.value.code == 1


def test_panel_too_large_is_rejected(T, h):
    """(2 n1 + 1)(2 n2 + 1) must fit the 32-bit bin index (ADVICE r1): rejected with an argument error, no allocation attempted."""
    with pytest.raises(T.TdsfsError) as e:
        h.set_panel(23170, 23170, True)   # 46341^2 = 2,147,488,281 > 2^31 - 1 = 2,147,483,647
    assert e.value.code == T.ERR_ARG
    h.set_panel(23169, 23169, True)       # 46339^2 = 2,147,302,921 fits
