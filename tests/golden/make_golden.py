#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/ from the UNMODIFIED reference.

Run in the build container only:   python tests/golden/make_golden.py
(needs /root/reference; the GPU box does not have it, the fixtures travel instead).

Fixtures written:
  chr1_counts.npz        compact form of data/chr1.pkl.bz2 (418,367 SNPs, uv/bv counts, annotation codes)
  ecb_chr1_{20kb,500kb,500snps}.csv   chromosome-"1" rows of the reference's SHIPPED outputs
                         data/ECBstats_*.csv (golden KATs, SURVEY.md section 4)
  chr1_ref_runs.npz      outputs of the reference class run HERE on chr1 (combined_scan 20 kb / 500 kb,
                         scan_perChr_bySNPs 500, scan_precomputed_BG 100 kb, missense-only scan, backgrounds)
  small_cases.json       seeded random data_dicts + the reference's outputs / raised exceptions for every
                         scanner, spectrum builder and likelihood (class and sims_scan twins)
  ingest_small.vcf.gz, ingest_small.popmap.txt, ingest_small.json
                         hand-built VCF exercising the ingest gates + reference make_data_dict_vcf output
  poisson_cases.json     seeded random data_dicts + the outputs of the first-generation script's Poisson window scan
                         (scripts/twoDSFS.py: calculate_2d_sfs with pseudo-counts, normalize_2d_sfs, calculate_p_window)
  ecb_subset.vcf.gz, ecb_subset.popmap.txt, ecb_subset.json
                         first contigs of vcf_pruned/ECB_LDpruned.vcf.gz with the header-derived popmap
                         (SURVEY.md section 9 Q1) + reference outputs at 20 kb / 500 kb / 500-SNP
"""
import bz2, csv, gzip, io, json, math, os, pickle, sys, contextlib
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from _ref_loader import load_class, load_sims, load_legacy, REF  # noqa: E402

RefClass = load_class()
sims = load_sims()


def jf(x):
    """JSON-able float/None (inf/nan allowed by python's json)."""
    if x is None:
        return None
    return float(x)


def res_to_list(res):
    out = []
    for k, v in res.items():
        out.append([k, {kk: (vv if isinstance(vv, (int, str)) or vv is None else jf(vv)) for kk, vv in v.items()}])
    return out


def sfs2d_to_list(d):
    return [[int(i), int(j), (int(v) if float(v).is_integer() else float(v))] for (i, j), v in d.items() if v != 0] + \
           [["nkeys", len(d)]]


def call(fn, *a, **k):
    """Run fn; return ('ok', value) or ('raises', ExceptionTypeName)."""
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            return "ok", fn(*a, **k)
    except Exception as e:  # noqa: BLE001 - we record the reference's exception type
        return "raises", type(e).__name__


# ----------------------------------------------------------------------------- chr1
def do_chr1():
    d = pickle.load(bz2.BZ2File(f"{REF}/data/chr1.pkl.bz2", "rb"))
    keys = list(d.keys())
    chrom = keys[0].split("-")[0]
    pos = np.array([int(k.split("-")[1]) for k in keys], dtype=np.int32)
    cnt = np.zeros((len(keys), 4), dtype=np.uint8)
    vocab, codes = {}, np.zeros(len(keys), dtype=np.uint8)
    for i, k in enumerate(keys):
        v = d[k]
        cnt[i, 0:2] = v["calls"]["uv"]
        cnt[i, 2:4] = v["calls"]["bv"]
        codes[i] = vocab.setdefault(v["annotation"], len(vocab))
    gaps = np.diff(pos.astype(np.int64), prepend=0)  # positions as uint16 gaps keep the file under 1 MB
    assert gaps.min() >= 1 and gaps.max() < 1 << 16
    np.savez_compressed(f"{HERE}/chr1_counts.npz", chrom=np.array(chrom), pos_delta=gaps.astype(np.uint16), cnt=cnt,
                        ann_code=codes, ann_vocab=np.array(sorted(vocab, key=vocab.get)))

    # shipped CSV rows for chromosome "1"
    for tag in ("20kb", "500kb", "500snps"):
        rows = list(csv.reader(open(f"{REF}/data/ECBstats_{tag}.csv")))
        hdr, body = rows[0], [r for r in rows[1:] if r[0] == "1"]
        with open(f"{HERE}/ecb_chr1_{tag}.csv", "w", newline="") as f:
            w = csv.writer(f)
            w.writerow(hdr[:10])
            for r in body:
                w.writerow(r[:10])
        print(tag, len(body), "rows")

    inst = RefClass("x", "y")  # defaults: uv/bv, 18/14, fold=True

    def pack(res, extra=("T2D_diff",)):
        n = len(res)
        out = dict(start=np.zeros(n, np.int64), end=np.zeros(n, np.int64), snp_count=np.zeros(n, np.int32))
        names = ["T2D", "T1D_pop1", "T1D_pop2", "new_term_pop1", "new_term_pop2"] + list(extra)
        for nm in names:
            out[nm] = np.full(n, np.nan)
            out[nm + "_none"] = np.zeros(n, bool)
        for i, (k, v) in enumerate(res.items()):
            s, e = k.split(" ")[1].split("-")
            out["start"][i], out["end"][i], out["snp_count"][i] = int(s), int(e), v["snp_count"]
            for nm in names:
                if v[nm] is None:
                    out[nm + "_none"][i] = True
                else:
                    out[nm][i] = v[nm]
        return out

    runs = {}
    with contextlib.redirect_stdout(io.StringIO()):
        for tag, W in (("c20k", 20000), ("c500k", 500000)):
            for k, v in pack(inst.combined_scan(d, W)).items():
                runs[f"{tag}_{k}"] = v
        for k, v in pack(inst.scan_perChr_bySNPs(d, 500)).items():
            runs[f"s500_{k}"] = v
        # whole-chromosome NORMALISED background, scan_precomputed_BG at 100 kb (class :1970-1983 usage)
        bg2 = inst.normalize_2d_sfs(inst.calculate_2d_sfs(d))
        b1 = inst.normalize_1d_sfs(inst.fold_1d_sfs(inst.calculate_1d_sfs(d, "uv", 18, None, None, None)))
        b2 = inst.normalize_1d_sfs(inst.fold_1d_sfs(inst.calculate_1d_sfs(d, "bv", 14, None, None, None)))
        for k, v in pack(inst.scan_precomputed_BG(d, 100000, bg2, b1, b2), extra=()).items():
            runs[f"p100k_{k}"] = v
        for k, v in pack(inst.scan_chooseChr(d, 250000, chrom), extra=()).items():
            runs[f"cc250k_{k}"] = v
        for k, v in pack(inst.scan_chooseChr_bySNPs(d, 1000, chrom), extra=()).items():
            runs[f"ccs1000_{k}"] = v
        # raw background spectra (bit-exact integer checks)
        raw2 = inst.calculate_2d_sfs(d)
        runs["bg2d"] = np.array([[raw2[(i, j)] for j in range(29)] for i in range(37)], dtype=np.int64)
        runs["bg1d_uv"] = np.array([inst.calculate_1d_sfs(d, "uv", 18, None, None, None)[i] for i in range(37)], dtype=np.int64)
        runs["bg1d_bv"] = np.array([inst.calculate_1d_sfs(d, "bv", 14, None, None, None)[i] for i in range(29)], dtype=np.int64)
        # variant_type filter (missense only), 500 kb
        instm = RefClass("x", "y", variant_type="missense_variant")
        st, r = call(instm.combined_scan, d, 500000)
        assert st == "ok", r
        for k, v in pack(r).items():
            runs[f"mis500k_{k}"] = v
        # position filter [5e6, 6e6] via ctor start/end (affects 2D spectra + 1D spectra)
        instp = RefClass("x", "y", start_position=5000000, end_position=6000000)
        st, r = call(instp.scan_chooseChr, d, 500000, chrom)
        runs["pos_status"] = np.array(st if st == "ok" else r)
        if st == "ok":
            for k, v in pack(r, extra=()).items():
                runs[f"pos500k_{k}"] = v
    np.savez_compressed(f"{HERE}/chr1_ref_runs.npz", **runs)
    print("chr1 done")


# ----------------------------------------------------------------------------- small random cases
def rand_dict(rng, chroms, n1, n2, nsnp, L, pops=("uv", "bv"), p_missing_pop=0.0, miss=0.1, anns=("A", "B"), hi_freq=0.2, force_first_mid=False):
    """Random data_dict in INSERTION order shuffled (the reference sorts)."""
    items = []
    for c in chroms:
        ps = rng.choice(np.arange(0 if rng.random() < 0.3 else 1, L), size=min(nsnp, L - 1), replace=False)
        for p in ps:
            calls = {}
            f = rng.random() ** 3 if rng.random() > hi_freq else 1 - rng.random() ** 3
            for pop, n in zip(pops, (n1, n2)):
                if rng.random() < p_missing_pop:
                    continue
                called = 2 * n - 2 * rng.binomial(n, miss)
                alt = int(rng.binomial(called, min(max(f + rng.normal(0, 0.1), 0), 1)))
                calls[pop] = (int(called - alt), alt)
            items.append((f"{c}-{int(p)}", {"segregating": ("A", "C"), "context": "-A-", "calls": calls,
                                           "annotation": str(rng.choice(anns))}))
    if force_first_mid:  # make the first SNP of every chromosome informative in both pops (sims_process_window path)
        for c in chroms:
            idx = min((i for i, it in enumerate(items) if it[0].startswith(c + "-")), key=lambda i: int(items[i][0].split("-")[1]))
            items[idx][1]["calls"] = {pops[0]: (2 * n1 - 1 - (n1 > 2), 1 + (n1 > 2)), pops[1]: (2 * n2 - 1, 1)}
    order = rng.permutation(len(items))
    return {items[i][0]: items[i][1] for i in order}


def dict_to_rows(d, pops):
    rows = []
    for k, v in d.items():
        c, p = k.split("-")
        r = [c, int(p)]
        for pop in pops:
            r.append(list(v["calls"][pop]) if pop in v["calls"] else None)
        r.append(v["annotation"])
        rows.append(r)
    return rows


def do_small():
    cases = []
    rng = np.random.default_rng(20241018)
    specs = [
        # name, chroms, n1, n2, nsnp/chrom, L, ctor kwargs, extras
        dict(name="two_chrom_dense", chroms=["chr2", "chr10"], n1=4, n2=3, nsnp=300, L=5000, W=[500, 2000], N=[25]),
        dict(name="sparse_windows_none", chroms=["c1", "c2", "c3"], n1=3, n2=3, nsnp=40, L=20000, W=[300, 1000], N=[7], miss=0.3),
        dict(name="missing_pop_records", chroms=["x"], n1=5, n2=4, nsnp=200, L=3000, W=[250], N=[20], p_missing_pop=0.15),
        dict(name="tiny_panel", chroms=["a", "b"], n1=2, n2=2, nsnp=150, L=2000, W=[100, 400], N=[10]),
        dict(name="big_panel", chroms=["k1", "k2"], n1=20, n2=25, nsnp=400, L=40000, W=[5000], N=[50], miss=0.05),
        dict(name="unfolded", chroms=["u1", "u2"], n1=4, n2=4, nsnp=200, L=4000, W=[500], N=[20], ctor=dict(fold=False)),
        dict(name="variant_filter", chroms=["v1", "v2"], n1=4, n2=4, nsnp=250, L=4000, W=[500], N=[20], ctor=dict(variant_type="A")),
        dict(name="pos_filter", chroms=["p1"], n1=4, n2=4, nsnp=300, L=6000, W=[500], N=[20], ctor=dict(start_position=1000, end_position=4000)),
        dict(name="hi_freq", chroms=["h1", "h2"], n1=6, n2=5, nsnp=250, L=5000, W=[700], N=[30], hi_freq=0.7),
        dict(name="first_snp_mid", chroms=["m1", "m2", "m3"], n1=4, n2=4, nsnp=200, L=3000, W=[400], N=[15], force_first_mid=True),
        dict(name="first_window_none", chroms=["f1"], n1=3, n2=3, nsnp=60, L=6000, W=[50], N=[5], miss=0.45),
    ]
    for sp in specs:
        pops = ("uv", "bv")
        d = rand_dict(rng, sp["chroms"], sp["n1"], sp["n2"], sp["nsnp"], sp["L"], pops=pops,
                      p_missing_pop=sp.get("p_missing_pop", 0.0), miss=sp.get("miss", 0.1), hi_freq=sp.get("hi_freq", 0.2),
                      force_first_mid=sp.get("force_first_mid", False))
        ctor = dict(pop1="uv", pop2="bv", pop1_size=sp["n1"], pop2_size=sp["n2"])
        ctor.update(sp.get("ctor", {}))
        mk = lambda: RefClass("x", "y", **ctor)  # noqa: E731 - fresh instance per call (methods mutate self)
        calls = []

        def rec(method, args, st, r, conv):
            calls.append(dict(method=method, args=args, status=st, result=(conv(r) if st == "ok" else r)))

        inst = mk()
        st, raw2 = call(inst.calculate_2d_sfs, d)
        rec("calculate_2d_sfs", [], st, raw2, sfs2d_to_list)
        one = {}
        for pop, n in ((ctor["pop1"], sp["n1"]), (ctor["pop2"], sp["n2"])):
            st, r = call(mk().calculate_1d_sfs, d, pop, n, ctor.get("start_position"), ctor.get("end_position"), ctor.get("variant_type"))
            rec("calculate_1d_sfs", [pop, n], st, r, lambda x: [[int(k), int(v)] for k, v in x.items()])
            one[pop] = r
            st, r2 = call(mk().fold_1d_sfs, r)
            rec("fold_1d_sfs", [pop], st, r2, lambda x: [[int(k), int(v)] for k, v in x.items()])
            one[pop + "_f"] = r2
        st, r = call(mk().normalize_2d_sfs, raw2)
        rec("normalize_2d_sfs", [], st, r, sfs2d_to_list)
        st, r = call(mk().count_snps, d, "A")
        rec("count_snps", ["A"], st, r, int)
        for W in sp["W"]:
            st, r = call(mk().combined_scan, d, W)
            rec("combined_scan", [W], st, r, res_to_list)
            for bgc in sp["chroms"][:2]:
                st, r = call(mk().scan_chooseChr, d, W, bgc)
                rec("scan_chooseChr", [W, bgc], st, r, res_to_list)
            st, r = call(mk().scan_chooseChr, d, W, "nope")
            rec("scan_chooseChr", [W, "nope"], st, r, res_to_list)
            # precomputed background = raw whole-dict spectra (counts) and normalised
            st, r = call(mk().scan_precomputed_BG, d, W, raw2, one["uv_f"], one["bv_f"])
            rec("scan_precomputed_BG_raw", [W], st, r, res_to_list)
            st_n, bgn = call(mk().normalize_2d_sfs, raw2)
            st_1, b1n = call(mk().normalize_1d_sfs, one["uv_f"])
            st_2, b2n = call(mk().normalize_1d_sfs, one["bv_f"])
            if st_n == st_1 == st_2 == "ok":
                st, r = call(mk().scan_precomputed_BG, d, W, bgn, b1n, b2n)
                rec("scan_precomputed_BG_norm", [W], st, r, res_to_list)
            st, r = call(mk().T2D_scan, d, raw2, W)
            rec("T2D_scan", [W], st, r, res_to_list)
            st, r = call(mk().T1D_scan, d, one["uv_f"], W, "uv", sp["n1"])
            rec("T1D_scan", [W, "uv", sp["n1"]], st, r, res_to_list)
            # sims twins (free functions, explicit args, no guards); background = first chromosome region, 1D UNFOLDED
            a = (ctor["pop1"], ctor["pop2"], sp["n1"], sp["n2"])
            st, sb2 = call(sims["calculate_2d_sfs"], d, *a, 0, sp["L"] // 2, None)
            st, sb1 = call(sims["calculate_1d_sfs"], d, a[0], a[2], 0, sp["L"] // 2, None)
            st, sb2b = call(sims["calculate_1d_sfs"], d, a[1], a[3], 0, sp["L"] // 2, None)
            st, r = call(sims["process_window"], d, sb2, sb1, sb2b, W, *a, None, None, None)
            rec("sims.process_window", [W, sp["L"] // 2], st, r, res_to_list)
            st, r = call(mk().sims_process_window, d, W, raw2, one["uv_f"], one["bv_f"])
            rec("sims_process_window", [W], st, r, res_to_list)
        for N in sp["N"]:
            st, r = call(mk().scan_perChr_bySNPs, d, N)
            rec("scan_perChr_bySNPs", [N], st, r, res_to_list)
            st, r = call(mk().scan_chooseChr_bySNPs, d, N, sp["chroms"][0])
            rec("scan_chooseChr_bySNPs", [N, sp["chroms"][0]], st, r, res_to_list)
        cases.append(dict(name=sp["name"], ctor=ctor, pops=list(pops), rows=dict_to_rows(d, pops), calls=calls))
        print(sp["name"], len(d), "snps", len(calls), "calls", [c["method"] for c in calls if c["status"] != "ok"])

    # direct likelihood KATs (None / inf / zero / float backgrounds)
    lk = []
    inst = RefClass("x", "y")
    r2 = np.random.default_rng(7)
    for t in range(40):
        nb = int(r2.integers(3, 30))
        fg = {i: int(v) for i, v in enumerate(r2.poisson(r2.choice([0.0, 0.3, 3.0, 40.0]), nb))}
        mode = t % 5
        if mode == 0:
            bg = {i: int(v) for i, v in enumerate(r2.poisson(50, nb))}
        elif mode == 1:
            bg = {i: float(v) for i, v in enumerate(r2.random(nb))}
        elif mode == 2:
            bg = {i: int(v) for i, v in enumerate(r2.poisson(0.7, nb))}  # zeros -> inf
        elif mode == 3:
            bg = dict(fg)  # identical -> 0.0
        else:
            bg = {i: 0 for i in range(nb)}  # B == 0 -> None
        st, r = call(inst.calculate_likelihood_1D, fg, bg)
        st2, rs = call(sims["calculate_likelihood_1D"], fg, bg)
        lk.append(dict(fg=list(fg.values()), bg=list(bg.values()), cls_status=st, cls=(jf(r) if st == "ok" else r),
                       sims_status=st2, sims=(jf(rs) if st2 == "ok" else rs)))
    # legacy Poisson score KATs (calculate_p, class :249-289)
    pk = []
    for t in range(12):
        nb = int(r2.integers(4, 40))
        fgp = {(i // 5, i % 5): int(v) for i, v in enumerate(r2.poisson(r2.choice([0.5, 4.0, 30.0]), nb))}
        bgp = {k: float(v) for k, v in zip(fgp, r2.random(nb))}
        for k in list(bgp)[:: 7]:
            bgp[k] = 0.0  # zero expectation bins are skipped (:282-283)
        tot = sum(bgp.values())
        bgp = {k: v / tot for k, v in bgp.items()}
        st, r = call(inst.calculate_p, fgp, bgp)
        assert st == "ok"
        pk.append(dict(fg=[[k[0], k[1], v] for k, v in fgp.items()], bg=[[k[0], k[1], v] for k, v in bgp.items()], value=jf(r)))
    json.dump(dict(cases=cases, likelihood=lk, poisson=pk), open(f"{HERE}/small_cases.json", "w"), allow_nan=True)
    print("small done")


# ----------------------------------------------------------------------------- ingest
VCF_SMALL = """##fileformat=VCFv4.2
##source=hand-built ingest fixture
#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\tS2\tX9\tS3\tS4\tS5\tS6
c1\t10\t.\tA\tG\t.\tPASS\tANN=G|missense_variant|MODERATE\tGT\t0/0\t0/1\t1/1\t1/1\t./.\t0|1\t1|0
c1\t20\t.\ta\tt\t.\t.\tPR\tGT:DP\t0/1:3\t1/1:9\t0/0:1\t./1:2\t0/.:4\t1:5\t0:7
c1\t30\t.\tAC\tG\t.\tPASS\tPR\tGT\t0/0\t0/1\t1/1\t1/1\t0/0\t0/1\t1/1
c1\t40\t.\tA\tG,T\t.\tPASS\tPR\tGT\t0/0\t0/1\t1/1\t1/1\t0/0\t0/1\t1/1
c1\t50\t.\tA\tG\t.\tq10\tPR\tGT\t0/0\t0/1\t1/1\t1/1\t0/0\t0/1\t1/1
c1\t60\t.\tC\tT\t.\tPASS\tANN=T|synonymous_variant\tDP:GT\t5:0/1\t5:1/2\t5:0/0\t5:2/2\t5:0/1/1\t5:10/1\t5:./.
c2\t5\t.\tG\tA\t.\tPASS\tPR\tGT\t1/1\t1/1\t1/1\t1/1\t1/1\t0/1\t1/1
c2\t5\t.\tG\tC\t.\tPASS\tPR\tGT\t0/0\t0/0\t0/0\t0/1\t0/0\t0/1\t0/0
c10\t7\t.\tT\tC\t.\t.\tX|intron_variant|Y\tGT\t0/1\t0/1\t0/1\t0/1\t0/1\t0/1\t0/1
c1\t5\t.\tN\tC\t.\t.\tPR\tGT\t0/1\t0/1\t0/1\t0/1\t0/1\t0/1\t0/1
c1\t70\t.\tG\tC\t.\tPASS\tPR\tGT\t0/0\t0/0\t0/0
"""
POPMAP_SMALL = "S1\tuv\nS2\tuv\nS3\tbv\nS4\tbv\nS5\tuv\nS6\tbv\nS7\tbv\nbadline\n"


def data_dict_json(d):
    return [[k, v["segregating"], v["context"], {p: list(c) for p, c in v["calls"].items()}, v["annotation"]] for k, v in d.items()]


def do_ingest():
    with gzip.open(f"{HERE}/ingest_small.vcf.gz", "wt") as f:
        f.write(VCF_SMALL)
    open(f"{HERE}/ingest_small.popmap.txt", "w").write(POPMAP_SMALL)
    inst = RefClass("x", "y")
    st, d = call(inst.make_data_dict_vcf, f"{HERE}/ingest_small.vcf.gz", f"{HERE}/ingest_small.popmap.txt")
    assert st == "ok", d
    st, ds = call(sims["make_data_dict_vcf"], f"{HERE}/ingest_small.vcf.gz", f"{HERE}/ingest_small.popmap.txt")
    assert st == "ok" and data_dict_json(ds) == data_dict_json(d)
    json.dump(dict(data_dict=data_dict_json(d)), open(f"{HERE}/ingest_small.json", "w"))

    # ECB subset: first 4 contigs of the shipped pruned VCF, header-derived popmap (SURVEY 9.Q1)
    src = gzip.open(f"{REF}/vcf_pruned/ECB_LDpruned.vcf.gz", "rt")
    out = gzip.open(f"{HERE}/ecb_subset.vcf.gz", "wt")
    contigs, samples = [], []
    for line in src:
        if line.startswith("##"):
            if not line.startswith("##contig"):
                out.write(line)
            continue
        if line.startswith("#"):
            samples = line.split()[9:]
            out.write(line)
            continue
        c = line.split("\t", 1)[0]
        if c not in contigs:
            if len(contigs) == 4:
                break
            contigs.append(c)
        out.write(line)
    out.close()
    with open(f"{HERE}/ecb_subset.popmap.txt", "w") as f:
        for s in samples:
            f.write(f"{s}\t{'bv' if s.startswith('EA') else 'uv'}\n")
    inst = RefClass("x", "y")
    st, d = call(inst.make_data_dict_vcf, f"{HERE}/ecb_subset.vcf.gz", f"{HERE}/ecb_subset.popmap.txt")
    assert st == "ok", d
    outj = dict(n_snps=len(d), first=data_dict_json({k: d[k] for k in list(d)[:50]}))
    # per-SNP counts for the whole subset (compact)
    outj["counts"] = [[k, list(v["calls"]["uv"]), list(v["calls"]["bv"])] for k, v in d.items()]
    for name, fn, arg in (("combined_20kb", "combined_scan", 20000), ("combined_500kb", "combined_scan", 500000),
                          ("bysnps_500", "scan_perChr_bySNPs", 500)):
        st, r = call(getattr(RefClass("x", "y"), fn), d, arg)
        outj[name] = dict(status=st, result=(res_to_list(r) if st == "ok" else r))
        print(name, st, len(r) if st == "ok" else r)
    json.dump(outj, open(f"{HERE}/ecb_subset.json", "w"), allow_nan=True)
    print("ingest done", len(d))


def do_poisson():
    """scripts/twoDSFS.py:211-463 run unmodified: unfolded 2D spectrum with a 1/total pseudo-count on every bin, background
    normalised over the interior, per-window sum of poisson.logpmf over the bins with a non-zero expectation."""
    L = load_legacy()
    rng = np.random.default_rng(20241007)
    cases = []
    specs = [  # chroms, n1, n2, snps per chrom, L, window, start, end, variant_type, background
        (["c2", "c10", "c1"], 4, 3, 220, 9000, 1000, None, None, None, "genome"),
        (["1"], 6, 5, 400, 30000, 2500, None, None, "A", "genome"),
        (["7", "x"], 3, 3, 90, 12000, 3000, 2000, 9000, None, "genome"),
        (["a", "b"], 5, 2, 150, 5000, 400, None, None, None, "other"),       # background from a different dict: zero-expectation bins
        (["s"], 2, 2, 12, 60000, 5000, None, None, None, "genome"),           # sparse: one-SNP windows (the int(x + 1/1) quirk)
        (["k1", "k2"], 8, 8, 700, 20000, 20000, None, None, None, "genome"),  # one big window per chromosome
    ]
    for chroms, n1, n2, nsnp, Lc, W, st, en, vt, bgk in specs:
        d = rand_dict(rng, chroms, n1, n2, nsnp, Lc, miss=0.05)
        src = d if bgk == "genome" else rand_dict(rng, chroms, n1, n2, max(nsnp // 3, 5), Lc, miss=0.05)
        bg = L["calculate_2d_sfs"](src, "uv", "bv", n1, n2, None, None, None)
        bgn = L["normalize_2d_sfs"](bg)
        res = L["calculate_p_window"](d, bgn, W, "uv", "bv", n1, n2, st, en, vt)
        cases.append(dict(n1=n1, n2=n2, W=W, start=st, end=en, variant_type=vt, rows=dict_to_rows(d, ("uv", "bv")),
                          bg_rows=None if bgk == "genome" else dict_to_rows(src, ("uv", "bv")),
                          bg_norm=[[k[0], k[1], jf(v)] for k, v in bgn.items()],
                          windows=[[k, jf(v["p_values"]), v["snp_count"]] for k, v in res.items()]))
    json.dump(dict(cases=cases), open(f"{HERE}/poisson_cases.json", "w"), allow_nan=True)
    print("poisson done", [len(c["windows"]) for c in cases])


if __name__ == "__main__":
    what = sys.argv[1:] or ["chr1", "small", "ingest", "poisson"]
    if "poisson" in what:
        do_poisson()
    if "chr1" in what:
        do_chr1()
    if "small" in what:
        do_small()
    if "ingest" in what:
        do_ingest()
