"""Shared helpers for the test-suite (fixture loading, tolerant comparison)."""
import csv
import json
import math
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL = 1e-9  # north-star tolerance: |d| <= 1e-9 * max(|T|, 1)


def close(a, b, rtol=RTOL):
    if a is None or b is None:
        return a is None and b is None
    if isinstance(a, str) or isinstance(b, str):
        return a == b
    a, b = float(a), float(b)
    if math.isnan(a) or math.isnan(b):
        return math.isnan(a) and math.isnan(b)
    if math.isinf(a) or math.isinf(b):
        return a == b
    return abs(a - b) <= rtol * max(abs(b), 1.0)


def load_small():
    return json.load(open(os.path.join(GOLDEN, "small_cases.json")))


def rows_to_dict(rows, pops):
    d = {}
    for r in rows:
        calls = {}
        for pop, c in zip(pops, r[2:2 + len(pops)]):
            if c is not None:
                calls[pop] = tuple(c)
        d[f"{r[0]}-{r[1]}"] = {"segregating": ("A", "C"), "context": "-A-", "calls": calls, "annotation": r[-1]}
    return d


def _chr1_pos(z):
    """chr1_counts.npz stores the (increasing) positions as uint16 gaps: it stays under 1 MB that way."""
    return np.cumsum(z["pos_delta"], dtype=np.int64).astype(np.int32)


def load_chr1_dict():
    z = np.load(os.path.join(GOLDEN, "chr1_counts.npz"))
    chrom = str(z["chrom"])
    vocab = [str(v) for v in z["ann_vocab"]]
    pos, cnt, ann = _chr1_pos(z), z["cnt"], z["ann_code"]
    d = {}
    for p, c, a in zip(pos.tolist(), cnt.tolist(), ann.tolist()):
        d[f"{chrom}-{p}"] = {"segregating": ("N", "N"), "context": "-N-", "calls": {"bv": (c[2], c[3]), "uv": (c[0], c[1])},
                             "annotation": vocab[a]}
    return d


def load_chr1_arrays():
    z = np.load(os.path.join(GOLDEN, "chr1_counts.npz"))
    return str(z["chrom"]), _chr1_pos(z), z["cnt"].astype(np.uint16), z["ann_code"], [str(v) for v in z["ann_vocab"]]


def load_ecb_csv(tag):
    """Shipped reference output rows (chromosome '1'): list of dict with None for NA/empty."""
    out = []
    with open(os.path.join(GOLDEN, f"ecb_chr1_{tag}.csv")) as f:
        for r in csv.DictReader(f):
            rec = {}
            for k, v in r.items():
                if k == "chromosome":
                    rec[k] = v
                elif k in ("window_start", "window_end", "snp_count"):
                    rec[k] = int(v)
                else:
                    rec[k] = None if v in ("NA", "") else float(v)
            out.append(rec)
    return out


def compare_result_lists(got, exp, what=""):
    """got: dict window->record (ours); exp: [[key, record], ...] from the reference."""
    gk = list(got.keys())
    ek = [k for k, _ in exp]
    assert gk == ek, f"{what}: window keys/order differ: {gk[:5]} vs {ek[:5]} (n={len(gk)} vs {len(ek)})"
    for k, rec in exp:
        g = got[k]
        assert list(g.keys()) == list(rec.keys()), f"{what} {k}: fields {list(g.keys())} vs {list(rec.keys())}"
        for f, v in rec.items():
            assert close(g[f], v), f"{what} {k} {f}: got {g[f]!r} expected {v!r}"
