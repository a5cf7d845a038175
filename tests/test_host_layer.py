"""CPU-only tests of the host logic of the drop-in layer: VCF ingest gates, dict <-> array conversion, filters."""
import json
import os

import numpy as np

from helpers import GOLDEN


def test_parse_vcf_matches_reference_ingest():
    import twoDSFS_class as K
    exp = json.load(open(os.path.join(GOLDEN, "ingest_small.json")))["data_dict"]
    d = K.parse_vcf_to_dict(os.path.join(GOLDEN, "ingest_small.vcf.gz"), os.path.join(GOLDEN, "ingest_small.popmap.txt"))
    got = [[k, list(v["segregating"]), v["context"], {p: list(c) for p, c in v["calls"].items()}, v["annotation"]] for k, v in d.items()]
    assert got == exp


def test_parse_ecb_subset_counts():
    import twoDSFS_class as K
    exp = json.load(open(os.path.join(GOLDEN, "ecb_subset.json")))
    d = K.parse_vcf_to_dict(os.path.join(GOLDEN, "ecb_subset.vcf.gz"), os.path.join(GOLDEN, "ecb_subset.popmap.txt"))
    assert [[k, list(v["calls"]["uv"]), list(v["calls"]["bv"])] for k, v in d.items()] == exp["counts"]


def test_cpp_and_python_ingest_agree():
    """parse_vcf_to_dict runs the text work in C++ (counts mode of csrc/vcf_pack.cpp); the Python loop is the same algorithm."""
    import twoDSFS_class as K
    for stem in ("ingest_small", "ecb_subset"):
        args = (os.path.join(GOLDEN, stem + ".vcf.gz"), os.path.join(GOLDEN, stem + ".popmap.txt"))
        a, b = K.parse_vcf_to_dict(*args), K._parse_vcf_to_dict_py(*args)
        assert a == b and list(a) == list(b) and all(list(a[k]["calls"]) == list(b[k]["calls"]) for k in a)


def test_snp_table_sorting_and_flags():
    from tdsfs_engine import SnpTable, filter_flags
    d = {"chr2-50": {"calls": {"a": (3, 1), "b": (2, 2)}, "annotation": "x"},
         "chr10-7": {"calls": {"a": (4, 0)}, "annotation": "y"},
         "chr2-5": {"calls": {"b": (1, 3)}, "annotation": "x"},
         "chr10-70": {"calls": {"a": (0, 4), "b": (4, 0)}, "annotation": "x"}}
    t = SnpTable.from_dict(d, "a", "b")
    assert t.chroms == ["chr10", "chr2"]  # string order, as the reference sorts
    assert t.keys == ["chr10-7", "chr10-70", "chr2-5", "chr2-50"]
    assert t.off.tolist() == [0, 2, 4] and t.pos.tolist() == [7, 70, 5, 50]
    assert t.cnt.tolist() == [[4, 0, 0, 0], [0, 4, 4, 0], [0, 0, 1, 3], [3, 1, 2, 2]]
    assert t.last_key_row == 1
    assert filter_flags(t, None, None, None) is None
    assert filter_flags(t, 6, 60, "x").tolist() == [0, 2, 2, 3]
    assert filter_flags(t, None, 60, None).tolist() == [3, 2, 3, 3]


def test_b32_layout_roundtrip():
    from tdsfs_pack import from_b32, to_b32
    rng = np.random.default_rng(0)
    rows = rng.integers(0, 2 ** 32, size=(70, 5), dtype=np.uint64).astype(np.uint32)
    buf = to_b32(rows)
    assert buf.size == 3 * 5 * 32
    assert buf[(40 // 32 * 5 + 3) * 32 + 40 % 32] == rows[40, 3]
    assert np.array_equal(from_b32(buf, 70, 5), rows)


def test_cpp_packer_matches_reference_ingest():
    """K0: the C++ packer applies the reference's ingest gates (positional poplist, FILTER/REF/ALT, duplicate keys,
    half calls as fix-ups) -- counts decoded from its 2-bit matrix equal the reference's data_dict."""
    from tdsfs_pack import pack_vcf
    for stem, pops in (("ingest_small", ("uv", "bv")), ("ecb_subset", ("uv", "bv"))):
        P = pack_vcf(os.path.join(GOLDEN, stem + ".vcf.gz"), os.path.join(GOLDEN, stem + ".popmap.txt"), *pops, nthreads=3)
        if stem == "ingest_small":
            exp = json.load(open(os.path.join(GOLDEN, stem + ".json")))["data_dict"]
            ref = {k: (calls.get("uv", [0, 0]), calls.get("bv", [0, 0]), ann) for k, _, _, calls, ann in exp}
        else:
            exp = json.load(open(os.path.join(GOLDEN, stem + ".json")))
            ref = {k: (u, b, "No annotation") for k, u, b in exp["counts"]}
        keys = [f"{P.chroms[c]}-{p}" for c in range(len(P.chroms)) for p in P.pos[P.off[c]:P.off[c + 1]].tolist()]
        assert sorted(keys) == sorted(ref)
        assert keys == sorted(ref, key=lambda k: (k.split("-")[0], int(k.split("-")[1])))
        cnt = P.counts()
        for i, k in enumerate(keys):
            assert cnt[i].tolist() == list(ref[k][0]) + list(ref[k][1]), (k, cnt[i], ref[k])
            assert P.ann[i] == ref[k][2]
    assert P.n_records == P.n + P.n_skipped or stem == "ingest_small"


def test_dictconv_c_path_equals_python_path():
    """csrc/dictconv.c (per-SNP loop of the dict -> array conversion in C) == the pure-Python conversion, errors included."""
    import pytest
    import tdsfs_engine as E
    from helpers import load_small, rows_to_dict
    conv = E._dictconv()
    if conv is None:
        pytest.skip("libtdsfs_dictconv.so not built")
    for case in load_small()["cases"]:
        d = rows_to_dict(case["rows"], case["pops"])
        a, b = E.SnpTable._from_dict_c(conv, d, "uv", "bv"), E.SnpTable._from_dict_py(d, "uv", "bv")
        for f in ("chroms", "keys", "n", "last_key_row", "pops"):
            assert getattr(a, f) == getattr(b, f), (case["name"], f)
        for f in ("pos", "cnt", "off"):
            assert np.array_equal(getattr(a, f), getattr(b, f)), (case["name"], f)
        assert list(a.ann) == list(b.ann)
    for bad, exc in (({"a-b-5": {"calls": {}}}, ValueError), ({"nodash": {"calls": {}}}, ValueError), ({"c-x": {"calls": {}}}, ValueError),
                     ({"c-5": {}}, KeyError)):
        for fn in (lambda: E.SnpTable._from_dict_c(conv, bad, "uv", "bv"), lambda: E.SnpTable._from_dict_py(bad, "uv", "bv")):
            with pytest.raises(exc):
                fn()
    assert E.SnpTable._from_dict_c(conv, {}, "a", "b").n == 0


def test_bench_checksums_do_not_depend_on_the_sharding():
    """bench.py's verify block: the order-independent checksums over all windows are the same however the windows are split
    over ranks (that is what makes the N = 1 / 2 / 4 / 8 bench lines comparable)."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    rng = np.random.default_rng(2)
    n = 5000
    res = dict(chrom=rng.integers(0, 32, n).astype(np.int32), start=(1 + 20000 * rng.integers(0, 4000, n)).astype(np.int64),
               snp_count=rng.integers(0, 700, n).astype(np.int32), n2d=rng.integers(0, 700, n).astype(np.int32),
               n1d_p1=rng.integers(0, 700, n).astype(np.int32), n1d_p2=rng.integers(0, 700, n).astype(np.int32),
               T2D=rng.normal(300, 50, n), T1D_p1=rng.normal(100, 20, n), T1D_p2=rng.normal(100, 20, n),
               flags=np.where(rng.random(n) < 0.05, 8, np.where(rng.random(n) < 0.02, 1, 0)).astype(np.uint8))
    res["snp_count"][res["flags"] == 8] = 0
    whole = bench.result_checksums(res, res["chrom"].astype(np.int64), 8, (1, 2, 4))
    for world in (2, 3, 8):
        cuts = np.sort(rng.choice(np.arange(1, n), size=world - 1, replace=False))
        parts = [bench.result_checksums({k: v[a:b] for k, v in res.items()}, res["chrom"][a:b].astype(np.int64), 8, (1, 2, 4))
                 for a, b in zip(np.concatenate([[0], cuts]), np.concatenate([cuts, [n]]))]
        tot = {k: sum(p[k] for p in parts) for k in whole}
        tot["int_checksum"] %= 1 << 64
        assert tot == whole
    # and they do depend on the content
    res["n2d"][17] += 1
    assert bench.result_checksums(res, res["chrom"].astype(np.int64), 8, (1, 2, 4))["int_checksum"] != whole["int_checksum"]


def test_bench_dump_outputs_are_float_and_capped(tmp_path):
    """bench.py --dump-outputs: one float64 .npy per result array, exact for the integer fields; above the byte cap the same
    seeded sample of windows on every run."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    rng = np.random.default_rng(4)
    n = 3000
    res = dict(chrom=rng.integers(0, 32, n).astype(np.int32), start=(1 + 20000 * rng.integers(0, 1 << 30, n)).astype(np.int64),
               T2D=rng.normal(300, 50, n), flags=rng.integers(0, 16, n).astype(np.uint8))
    bench.write_outputs(str(tmp_path / "all"), res, 7)
    for k, v in res.items():
        got = np.load(tmp_path / "all" / f"{k}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, v)
    assert np.array_equal(np.load(tmp_path / "all" / "window_index.npy"), np.arange(n))
    cap = 8 * (len(res) + 1) * 500
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), res, 7, cap_bytes=cap)
    idx = np.load(tmp_path / "a" / "window_index.npy")
    assert len(idx) == 500 and np.all(np.diff(idx) > 0)
    assert np.array_equal(idx, np.load(tmp_path / "b" / "window_index.npy"))
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) < cap + 1024 * (len(res) + 1)
    assert np.array_equal(np.load(tmp_path / "a" / "start.npy"), res["start"][idx.astype(np.int64)])
