#!/usr/bin/env python
"""Small scans that touch every kernel of the hot path, for compute-sanitizer (one tool per gpurun call):
  compute-sanitizer --tool racecheck|synccheck|memcheck python tools/sanitize_small.py
k1_fused (plain + generic instantiation, narrow + wide records, fixed-bp + fixed-SNP windows, chunked upload, flags),
k3_finish, k3_score_small (G = 1, 2, 4) + k3_score_large, k2_bounds_*, k_finalize_counts, k1_counts,
the Poisson walk.  Results are compared with the CPU oracle so that a sanitizer-only failure mode cannot hide."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "2dsfs-scan_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import sfs_oracle as O  # noqa: E402
import tdsfs_capi as T  # noqa: E402
from test_gpu_capi_parity import compare_scan, random_panel  # noqa: E402


def main():
    rng = np.random.default_rng(1)
    done = []
    for n1, n2, S, C, L, W, N in ((40, 33, 6000, 3, 120000, 4000, 150), (6, 5, 2500, 2, 50000, 3000, 40)):
        G, w1, w2, pos, off = random_panel(rng, S, n1, n2, C, L)
        cnt = O.unpack_counts(G, w1, w2, n1, n2, S)
        for chunk_kb in (None, "16"):
            if chunk_kb:
                os.environ["TDSFS_UPLOAD_CHUNK_KB"] = chunk_kb
            else:
                os.environ.pop("TDSFS_UPLOAD_CHUNK_KB", None)
            h = T.Handle(0)
            h.set_panel(n1, n2, True)
            h.load_genotypes(G, S, w1, w2, n1, n2, pos, off)
            for mode, bg in ((T.BG_GENOME, "genome"), (T.BG_PER_CHROM, "per_chrom")):
                h.plan(W)
                h.background(mode)
                h.finalize_background()
                res = h.scan(W)
                assert h.scan_info()[0]
                compare_scan(T, res, O.scan_arrays(cnt, pos, off, n1, n2, W=W, bg=bg))
                h.plan(N, snp_mode=True)
                h.background(mode)
                h.finalize_background()
                compare_scan(T, h.scan(N, snp_mode=True), O.scan_arrays(cnt, pos, off, n1, n2, N=N, bg=bg), snp_mode=True)
                done.append(("fused", n1, chunk_kb, bg))
            h.close()
        # table scorer (no plan), group widths, large windows, counts entry, wide records
        for g in ("1", "2", "4"):
            os.environ["TDSFS_SCORE_G"] = g
            os.environ["TDSFS_REC_WIDE"] = "1" if g == "2" else ""
            if not os.environ["TDSFS_REC_WIDE"]:
                os.environ.pop("TDSFS_REC_WIDE")
            h = T.Handle(0)
            h.set_panel(n1, n2, True)
            h.load_genotypes(G, S, w1, w2, n1, n2, pos, off)
            h.background(T.BG_PER_CHROM)
            h.finalize_background()
            compare_scan(T, h.scan(W), O.scan_arrays(cnt, pos, off, n1, n2, W=W))
            compare_scan(T, h.scan(20 * W), O.scan_arrays(cnt, pos, off, n1, n2, W=20 * W))
            h.load_counts(cnt.astype(np.uint16), pos, off)
            compare_scan(T, h.run_bp(T.BG_GENOME, W), O.scan_arrays(cnt, pos, off, n1, n2, W=W, bg="genome"))
            h.close()
            done.append(("table", n1, g))
        os.environ.pop("TDSFS_SCORE_G", None)
        # Poisson walk
        R2 = 2 * n2 + 1
        bgc = np.bincount(cnt[:, 1] * R2 + cnt[:, 3], minlength=(2 * n1 + 1) * R2).astype(np.float64)
        bgc[0] = 0
        bgc += 1.0 / bgc.sum()
        q = bgc / bgc[1:-1].sum()
        h = T.Handle(0)
        h.set_panel(n1, n2, False)
        h.load_genotypes(G, S, w1, w2, n1, n2, pos, off)
        h.background(T.BG_NONE)
        h.set_poisson_background(q)
        res = h.scan_poisson(W)
        live = np.flatnonzero((res["flags"] & T.F_EMPTY) == 0)
        assert len(live) and np.all(np.isfinite(res["T2D"][live]))
        h.close()
        done.append(("poisson", n1))
    print("sanitize_small: %d scan groups ok" % len(done))


if __name__ == "__main__":
    main()
