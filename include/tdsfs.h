/*
 * tdsfs.h -- C ABI of libtdsfs.so: the B200 (sm_100a) implementation of the 2DSFS-scan hot path.
 *
 * The reference (uricchio/2DSFS-scan) has no FFI; its boundary is the Python surface of
 * scripts/src/twoDSFS_class.py and scripts/sims_scan.py (paths below are relative to the reference
 * repository).  Every entry point here names the reference code whose body it replaces.  The Python
 * drop-in layer (2dsfs-scan_b200/twoDSFS_class.py, sims_scan.py) binds these with ctypes; INTEGRATION.md
 * shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - return 0 on success, non-zero (TDSFS_ERR_*) otherwise; tdsfs_last_error() gives a thread-local message.
 *   - input pointers may be HOST or DEVICE memory (detected with cudaPointerGetAttributes); device inputs are
 *     adopted without a copy and must outlive the scan.  Output pointers are caller-owned HOST buffers.
 *   - the library owns every device allocation behind the handle; it never returns memory it allocated.
 *   - calls are synchronous unless stated (they synchronise the handle's stream before returning);
 *     one handle = one GPU, not re-entrant.
 *   - there is NO CPU fallback: without a CUDA device tdsfs_create fails.
 */
#ifndef TDSFS_H
#define TDSFS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tdsfs_ctx tdsfs_t;

enum {
  TDSFS_OK = 0,
  TDSFS_ERR_ARG = 1,    /* bad argument / buffer too small */
  TDSFS_ERR_CUDA = 2,   /* CUDA runtime error (message has the cudaError string) */
  TDSFS_ERR_STATE = 3,  /* call order violated (e.g. scan before background) */
  TDSFS_ERR_RANGE = 4,  /* an allele count exceeds 2n of the declared panel: the reference raises KeyError
                           (twoDSFS_class.py:433) for the same input */
  TDSFS_ERR_RETRY = 5   /* asynchronous pass only: a SNP did not fit the 4-byte per-SNP record; the handle has switched
                           to 8-byte records and the pass must be run again (synchronous calls and tdsfs_run_bp retry
                           by themselves) */
};

/* result flags (per candidate window) */
enum {
  TDSFS_F_T2D_NONE = 1,    /* calculate_likelihood_2D returned None (twoDSFS_class.py:645-647, :668-670) */
  TDSFS_F_T1D_P1_NONE = 2, /* calculate_likelihood_1D returned None for pop1 (:497-499, :520-522) */
  TDSFS_F_T1D_P2_NONE = 4,
  TDSFS_F_EMPTY = 8,       /* window holds no SNP: the reference never emits it (:902 `if window_data`) */
  TDSFS_F_SKIPPED = 16     /* fixed-SNP window whose 2D spectrum sums to 0 (:1496) */
};

/* background modes for tdsfs_background() */
enum {
  TDSFS_BG_NONE = 0,      /* keys only; background supplied later with tdsfs_set_background (scan_precomputed_BG :1161) */
  TDSFS_BG_PER_CHROM = 1, /* every chromosome its own background (combined_scan :809-825, scan_perChr_bySNPs :1450-1460) */
  TDSFS_BG_GENOME = 2,    /* one background over all loaded SNPs (whole-genome usage :1970-1981; the north-star mode) */
  TDSFS_BG_CHROM = 3      /* background = one chromosome (scan_chooseChr :1021-1034) */
};

/* Sparse correction for calls the 2-bit code cannot hold (half calls './1', haploid '1', ...):
 * the sample is stored as MISSING and (dref, dalt) is added to its population's counts, reproducing the
 * per-character counting of make_data_dict_vcf (twoDSFS_class.py:128-129).  Sorted by snp. */
typedef struct {
  int64_t snp;
  int32_t pop; /* 0 = pop1, 1 = pop2 */
  int32_t dref;
  int32_t dalt;
} tdsfs_fixup_t;

/* Struct-of-arrays result, caller-owned host buffers of capacity >= the candidate count
 * (tdsfs_candidates_bp / _snp).  Replaces the dict of dicts built at twoDSFS_class.py:937-945.
 * Any member may be NULL (skipped). */
typedef struct {
  int32_t* chrom;     /* chromosome index (order of chrom_off) */
  int64_t* start;     /* label start: 1 + k*W (fixed-bp) / first SNP pos or previous end + 1 (fixed-SNP, :1527/:1535) */
  int64_t* end;       /* label end: start + W - 1 / last SNP pos */
  int32_t* snp_count; /* count_snps (:291-302) */
  int32_t* n2d;       /* N of the 2D likelihood = SNPs in interior bins (:642) */
  int32_t* n1d_p1;
  int32_t* n1d_p2;
  double* T2D;        /* 2*(ll_fg - ll_bg), +inf when a populated bin has zero background */
  double* T1D_p1;
  double* T1D_p2;
  uint8_t* flags;     /* TDSFS_F_* */
} tdsfs_result_t;

/* ---- lifetime ------------------------------------------------------------------------------------------ */
int tdsfs_create(int device, tdsfs_t** out);
void tdsfs_destroy(tdsfs_t* ctx);
const char* tdsfs_last_error(void);
/* Run the handle's work on an existing CUDA stream (cudaStream_t as void*; NULL = the handle's own stream). */
int tdsfs_set_stream(tdsfs_t* ctx, void* cuda_stream);
/* sync = 0: tdsfs_background / tdsfs_finalize_background / tdsfs_scan_*(out = NULL) only enqueue work on the stream
 * and return; the caller synchronises (used to time the whole pass on the device and to chain the all-reduce). */
int tdsfs_set_sync(tdsfs_t* ctx, int sync);

/* Declared diploid panel sizes -> spectrum shape (2*n1+1) x (2*n2+1); fold = joint minor-allele fold.
 * Replaces the constructor state pop1_size/pop2_size/fold (twoDSFS_class.py:21-33). */
int tdsfs_set_panel(tdsfs_t* ctx, int32_t n1, int32_t n2, int32_t fold);

/* ---- data (the data_dict, twoDSFS_class.py:132-134, in array form) ---------------------------------------
 * SNPs sorted by (chromosome, position); chrom_off[C+1] row offsets of the chromosomes (host memory).
 * snp_flags (optional, S bytes): bit0 = SNP passes the spectrum filters (start/end position :179-182 and
 * variant_type :185-187), bit1 = SNP counts in snp_count (count_snps :298-301).  NULL = all pass. */

/* Counts-level entry: cnt[S][4] = (ref1, alt1, ref2, alt2), the 'calls' tuples of the data_dict. */
int tdsfs_load_counts(tdsfs_t* ctx, const uint16_t* cnt, int64_t S, const int32_t* pos, const int64_t* chrom_off,
                      int32_t C, const uint8_t* snp_flags);

/* Genotype-level entry: 2-bit-per-call matrix, stored as bit planes.  Per SNP: RW = words1 + words2 uint32 words; a
 * population is words/2 pairs (lo word, hi word) of 32 samples each: bit b of the lo / hi word of pair g is the low /
 * high bit of the code of sample 32g + b.  pop1 pairs then pop2 pairs, each population zero padded to a whole pair
 * (words1, words2 even: words = 2 * ceil(samples / 32)).
 * Memory layout "B32" (block transposed): SNPs in blocks of 32; word w of SNP s at uint32 index
 * ((s / 32) * RW + w) * 32 + s % 32; the buffer holds ceil(S / 32) whole blocks (rows beyond S zero).
 * Codes: 0 = 0/0, 1 = 0/1, 3 = 1/1, 2 = missing, so #missing = popcount(hi & ~lo), alt = popcount(all words) - #missing,
 * ref = 2 * (samples - #missing) - alt.  ns1/ns2 = number of sample columns in each block.
 * Replaces the per-sample counting loop of make_data_dict_vcf (:118-130).  Host G is uploaded in chunks
 * asynchronously; the upload overlaps the count kernel of tdsfs_background. */
int tdsfs_load_genotypes(tdsfs_t* ctx, const void* G, int64_t S, int32_t words1, int32_t words2, int32_t ns1,
                         int32_t ns2, const int32_t* pos, const int64_t* chrom_off, int32_t C,
                         const tdsfs_fixup_t* fixups, int64_t n_fixups, const uint8_t* snp_flags);

/* ---- spectra + background --------------------------------------------------------------------------------
 * Derives every SNP's folded 2D bin and raw 1D alt counts (calculate_2d_sfs :190-217, calculate_1d_sfs :427-433)
 * and accumulates the integer background spectra of the requested mode.  bg_chrom: chromosome index for
 * TDSFS_BG_CHROM.  [bg_pos_lo, bg_pos_hi] restricts the SNPs that enter the background (sims_scan.py:664-666
 * uses 0..500000); pass -1, -1 for no restriction. */
int tdsfs_background(tdsfs_t* ctx, int32_t mode, int32_t bg_chrom, int64_t bg_pos_lo, int64_t bg_pos_hi);

/* Number of background groups (C for PER_CHROM, else 1) and the packed device histogram
 * [group][ (2n1+1)(2n2+1) | 2n1+1 | 2n2+1 ] of uint32 counts, for an in-place all-reduce (sum) across GPUs
 * before tdsfs_finalize_background.  n_words = total uint32 words. */
int tdsfs_background_device(tdsfs_t* ctx, void** dev_ptr, int64_t* n_words, int32_t* n_groups);

/* ---- peer-memory exchange of the background (multi-GPU, one process per GPU on one NVLink/NVSwitch node) -----
 * The genome-wide background of a chromosome-sharded scan is the SUM of the ranks' histograms; the reference
 * computes it in one process (calculate_2d_sfs on the whole data_dict, :809-825), so this step has no reference
 * counterpart.  Instead of a library all-reduce, every rank maps every other rank's histogram (CUDA IPC) and one
 * kernel per rank pulls its slice of all histograms over NVLink, sums it and pushes the sum back into all of them,
 * between two flag barriers in peer memory.  Protocol, collectively on all ranks:
 *   tdsfs_background(...)                       once, so that the histogram exists (single group: GENOME / CHROM)
 *   tdsfs_peer_export(ctx, rank, world, blob)   fills blob[TDSFS_PEER_BLOB_BYTES]; exchange blobs out of band
 *   tdsfs_peer_import(ctx, blobs)               blobs = world x TDSFS_PEER_BLOB_BYTES in rank order
 *   per scan: tdsfs_background -> tdsfs_peer_reduce_finalize -> tdsfs_scan_*
 *   tdsfs_peer_close(ctx)                       on every rank BEFORE any rank changes its panel or is destroyed
 * The exchange is asynchronous on the handle's stream; all ranks must call it the same number of times.  A rank that
 * never arrives makes the others flag TDSFS_ERR_CUDA (tdsfs_check) after ~60 s (TDSFS_PEER_TIMEOUT_S), not hang. */
#define TDSFS_PEER_BLOB_BYTES 192
#define TDSFS_PEER_MAX_RANKS 16
int tdsfs_peer_export(tdsfs_t* ctx, int32_t rank, int32_t world, void* blob);
int tdsfs_peer_import(tdsfs_t* ctx, const void* blobs);
/* The same call as tdsfs_peer_reduce_finalize: besides the all-reduce it builds the ln tables, so a
 * tdsfs_finalize_background that follows is a no-op unless tdsfs_background_device was called in between. */
int tdsfs_peer_allreduce_background(tdsfs_t* ctx);
/* The exchange and tdsfs_finalize_background in ONE launch per rank: barrier, pull / sum / push of this rank's slice,
 * barrier, then the ln tables of the complete local histogram.  A tdsfs_finalize_background that follows is a no-op
 * unless tdsfs_background_device was called in between. */
int tdsfs_peer_reduce_finalize(tdsfs_t* ctx);
int tdsfs_peer_close(tdsfs_t* ctx);

/* Copy one group's integer spectra to the host: sfs2d[(2n1+1)*(2n2+1)] row-major (i,j) = calculate_2d_sfs,
 * sfs1d_p1[2n1+1] / sfs1d_p2[2n2+1] = calculate_1d_sfs (unfolded).  Any pointer may be NULL. */
int tdsfs_get_background(tdsfs_t* ctx, int32_t group, uint64_t* sfs2d, uint64_t* sfs1d_p1, uint64_t* sfs1d_p2);

/* Precomputed background (scan_precomputed_BG :1161, sims_scan.process_window :451): b2d[(2n1+1)(2n2+1)] and,
 * per population, the values bg[k] seen by the folded foreground keys k = 0..n (n+1 doubles).  Counts or
 * normalised floats.  All chromosomes are scored against it. */
int tdsfs_set_background(tdsfs_t* ctx, const double* b2d, const double* b1d_p1, const double* b1d_p2);

/* Build the log tables the scorer reads (ln b_k, interior totals B).  Call after tdsfs_background (+ all-reduce)
 * or tdsfs_set_background. */
int tdsfs_finalize_background(tdsfs_t* ctx);

/* ---- scans -----------------------------------------------------------------------------------------------
 * Fixed-bp windows (window walk :843-949: window index (pos-1)//W per chromosome, empty windows flagged
 * TDSFS_F_EMPTY) and fixed-SNP windows (:1515-1535: full chunks of N SNPs, partial tail dropped).
 * `out` may be NULL: results then stay on the device (tdsfs_fetch_results copies them later); cap = capacity of
 * the out arrays; *n_windows = number of candidate windows written. */
/* Optional: launch the window-boundary kernel NOW on a side stream (it depends on positions only), so that it overlaps
 * tdsfs_background and the multi-GPU all-reduce; the next tdsfs_scan_* of the same size waits for it instead of launching it. */
int tdsfs_plan_bp(tdsfs_t* ctx, int64_t W);
int tdsfs_plan_snp(tdsfs_t* ctx, int64_t N);
int tdsfs_candidates_bp(tdsfs_t* ctx, int64_t W, int64_t* n_candidates);
int tdsfs_candidates_snp(tdsfs_t* ctx, int64_t N, int64_t* n_candidates);
int tdsfs_scan_bp(tdsfs_t* ctx, int64_t W, tdsfs_result_t* out, int64_t cap, int64_t* n_windows);
int tdsfs_scan_snp(tdsfs_t* ctx, int64_t N, tdsfs_result_t* out, int64_t cap, int64_t* n_windows);
int tdsfs_fetch_results(tdsfs_t* ctx, tdsfs_result_t* out, int64_t cap, int64_t* n_windows);

/* Synchronise the stream and report deferred device-side errors (TDSFS_ERR_RANGE) after asynchronous calls. */
int tdsfs_check(tdsfs_t* ctx);

/* One-call convenience used by the end-to-end benchmark: background(mode) -> finalize -> scan_bp. */
int tdsfs_run_bp(tdsfs_t* ctx, int32_t bg_mode, int64_t W, tdsfs_result_t* out, int64_t cap, int64_t* n_windows);

/* Legacy Poisson composite score of every fixed-bp window, the first-generation script's calculate_p_window
 * (scripts/twoDSFS.py:385-463; the class copy :304-393 cannot run): per window the UNFOLDED 2D spectrum keyed by raw alt
 * counts (twoDSFS.py:211-303: SNPs with both alt counts 0 skipped, a pseudo-count 1/total added to every bin), S_w = the sum
 * of all its bins, and the sum over the bins with S_w q != 0 of poisson.logpmf(int(count), S_w q) (:336-374).
 * q2d[(2n1+1)(2n2+1)] = the normalised background (normalize_2d_sfs :324-334).  Needs tdsfs_set_panel(..., fold = 0) and
 * tdsfs_background (any mode: it writes the per-SNP bins).  Results: T2D = the score, n2d = SNPs counted in the spectrum,
 * snp_count as in the other scans; the 1D fields are zero. */
int tdsfs_set_poisson_background(tdsfs_t* ctx, const double* q2d);
int tdsfs_scan_poisson_bp(tdsfs_t* ctx, int64_t W, tdsfs_result_t* out, int64_t cap, int64_t* n_windows);

/* One whole pass, asynchronous on the handle's stream: plan -> count kernel -> (peer exchange +) ln tables -> finish
 * kernel, results left on the device (tdsfs_fetch_results), deferred errors in tdsfs_check.  Called repeatedly with the
 * same arguments on device-resident data it captures the pass as a CUDA graph on the second call and replays it afterwards.
 * With the peer exchange mapped (tdsfs_peer_import) the exchange is part of the pass: every rank calls it the same number
 * of times. */
int tdsfs_step_bp(tdsfs_t* ctx, int32_t bg_mode, int64_t W);

/* Spectra of one scanned window (calculate_2d_sfs / calculate_1d_sfs on window_data): dense outputs, any NULL. */
int tdsfs_window_spectra(tdsfs_t* ctx, int64_t window, uint64_t* sfs2d, uint64_t* sfs1d_p1, uint64_t* sfs1d_p2);

/* ---- per-window diversity: Hudson FST, pi, dxy (no reference counterpart; DESIGN.md section 7) ------------------
 * Over the candidate windows of (size, mode), in the list and order of tdsfs_scan_* of that size, from the loaded data
 * alone (no background, no scan).  A SNP enters a window's sums iff it passes the spectrum filters (snp_flags bit0) and
 * n_i = ref_i + alt_i >= 2 in both populations (called alleles, fix-ups applied).  Per SNP, in fp64:
 *   pi_i = 2 ref_i alt_i / (n_i (n_i - 1)),   dxy = (ref_1 alt_2 + alt_1 ref_2) / (n_1 n_2)
 * pi_p1 / pi_p2 / dxy are SUMS over the entered (variant) sites, not per-bp values: dividing by a callable length is the
 * caller's business.  fst = 1 - (pi_p1 + pi_p2) / (2 dxy), Hudson's estimator as a ratio of averages (Bhatia et al. 2013,
 * eq. 10), NaN when dxy == 0.  The sums run in a fixed order that depends on the window's rows alone, so results are
 * bitwise equal for the counts and the genotype entry and for any sharding that keeps windows whole.
 * The call keeps its own window arrays and results: a pending plan, the scan's results and the step graph are untouched.
 * out == NULL: enqueue only (honours tdsfs_set_sync(0)); tdsfs_fetch_diversity copies the results later. */
typedef struct {            /* caller-owned host SoA, capacity >= tdsfs_candidates_bp / _snp; any member may be NULL */
  int32_t* chrom;           /* as tdsfs_result_t */
  int64_t* start;
  int64_t* end;
  int32_t* snp_count;       /* count_snps, as tdsfs_result_t */
  uint8_t* flags;           /* TDSFS_F_EMPTY */
  int32_t* n_sites;         /* SNPs that entered the sums */
  double* pi_p1;
  double* pi_p2;
  double* dxy;
  double* fst;              /* NaN when dxy == 0 */
} tdsfs_diversity_t;
int tdsfs_diversity_bp(tdsfs_t* ctx, int64_t W, tdsfs_diversity_t* out, int64_t cap, int64_t* n_windows);
int tdsfs_diversity_snp(tdsfs_t* ctx, int64_t N, tdsfs_diversity_t* out, int64_t cap, int64_t* n_windows);
int tdsfs_fetch_diversity(tdsfs_t* ctx, tdsfs_diversity_t* out, int64_t cap, int64_t* n_windows);

/* ---- per-window neutrality: Watterson's theta, Tajima's D per population (no reference counterpart; DESIGN.md 7) ---
 * Same windows, spectrum filter (snp_flags bit0) and counts (n_i = ref_i + alt_i called alleles, fix-ups applied) as
 * tdsfs_diversity_*.  Per window and population i, over the rows that pass the filter:
 *   n_seg_p<i>     S_i, rows with ref_i > 0 and alt_i > 0: segregating in population i, whatever the other population has;
 *   n_max_p<i>     the largest n_i (0 when no row passes);
 *   theta_pi_p<i>  the sum over rows with n_i >= 2 of 2 ref_i alt_i / (n_i (n_i - 1)) (fp64, exact integer numerator and
 *                  denominator, one rounded division), in the summation order of tdsfs_diversity_*.  It differs from that
 *                  call's pi_p<i> only on rows where the other population has n < 2, which pi_p<i> leaves out;
 *   theta_w_p<i>   S_i / a1(n_max_i), a1(n) = sum_{k=1}^{n-1} 1/k summed in ascending k; NaN when n_max_i < 2;
 *   tajima_d_p<i>  (theta_pi - theta_w) / sqrt(e1 S + e2 S (S - 1)), Tajima's (1989) constants at n = n_max_i:
 *                  a2 = sum_{k=1}^{n-1} 1/k^2, b1 = (n+1) / (3(n-1)), b2 = 2(n^2+n+3) / (9n(n-1)), c1 = b1 - 1/a1,
 *                  c2 = b2 - (n+2)/(a1 n) + a2/a1^2, e1 = c1/a1, e2 = c2/(a1^2 + a2); NaN when S_i < 3 or the variance
 *                  term is not > 0 (n_max = 2 makes e1 = e2 = 0).
 * This is scikit-allel's tajima_d (min_sites = 3) on the window's rows, with absolute theta: dividing by a callable length
 * is the caller's business.  The per-window n keeps results a function of the window's rows alone (bitwise equal for the
 * counts and the genotype entry and for any sharding that keeps windows whole); a caller who wants another n recomputes D
 * from n_seg, n_max and theta_pi.  Own window arrays and results, as tdsfs_diversity_*: neither call, a pending plan, the
 * scan's results nor the step graph disturbs the other.
 * out == NULL: enqueue only (honours tdsfs_set_sync(0)); tdsfs_fetch_neutrality copies the results later. */
typedef struct {            /* caller-owned host SoA, capacity >= tdsfs_candidates_bp / _snp; any member may be NULL */
  int32_t* chrom;           /* as tdsfs_result_t */
  int64_t* start;
  int64_t* end;
  int32_t* snp_count;       /* count_snps, as tdsfs_result_t */
  uint8_t* flags;           /* TDSFS_F_EMPTY */
  int32_t* n_seg_p1;        /* S_1 */
  int32_t* n_seg_p2;        /* S_2 */
  int32_t* n_max_p1;
  int32_t* n_max_p2;
  double* theta_pi_p1;
  double* theta_pi_p2;
  double* theta_w_p1;       /* NaN when n_max_p1 < 2 */
  double* theta_w_p2;
  double* tajima_d_p1;      /* NaN when S_1 < 3 or the variance term is not > 0 */
  double* tajima_d_p2;
} tdsfs_neutrality_t;
int tdsfs_neutrality_bp(tdsfs_t* ctx, int64_t W, tdsfs_neutrality_t* out, int64_t cap, int64_t* n_windows);
int tdsfs_neutrality_snp(tdsfs_t* ctx, int64_t N, tdsfs_neutrality_t* out, int64_t cap, int64_t* n_windows);
int tdsfs_fetch_neutrality(tdsfs_t* ctx, tdsfs_neutrality_t* out, int64_t cap, int64_t* n_windows);

/* ---- per-window Weir and Cockerham (1984) FST from the genotype calls (no reference counterpart; DESIGN.md 7) -------
 * Same windows, order and spectrum filter as tdsfs_diversity_*, for data loaded with tdsfs_load_genotypes only: the counts
 * entry has no heterozygote counts (TDSFS_ERR_STATE).  Per row, counts come from the 2-bit codes alone: calls held as
 * fix-ups (half calls, haploid calls, multi-allelic digits) count as missing.  For population i, n_i = called diploids
 * (ns_i - #missing), x_i = their alt alleles, h_i = their heterozygotes (code 1); N = n1 + n2, X = x1 + x2, H = h1 + h2,
 * D = x1 n2 - x2 n1.  The variance components summed over both alleles, each an exact int64 numerator over an exact int64
 * denominator, converted to fp64 and divided once (round to nearest):
 *   a = [D^2 (N-1) - n1 n2 (X(2N-X) - N H)] / [4 n1^2 n2^2 (N-2)]
 *   b = [n1 n2 (X(2N-X) - 2(N-1) H) - D^2] / [2 n1 n2 N (N-2)]
 *   c = H / N
 * a and b enter a window's sums for the rows that pass the filter (snp_flags bit0, read directly: no fix-up is applied)
 * with n1 >= 1, n2 >= 1 and N >= 3 (n_sites counts these rows); c for every row that passes the filter with N >= 1.
 * This is scikit-allel's weir_cockerham_fst (r = 2) summed over both alleles, with windowed_weir_cockerham_fst's nansum:
 * it gives NaN for a and b exactly on the rows left out here.  fst = a / ((a + b) + c), NaN when that denominator is 0;
 * it can be negative.  The sums run in the order of tdsfs_diversity_*, so results are bitwise equal for any sharding that
 * keeps windows whole.  Panels with more than 4000 samples in a population (the int64 terms would overflow) give
 * TDSFS_ERR_ARG.  Own window arrays and results, as tdsfs_diversity_*.
 * out == NULL: enqueue only (honours tdsfs_set_sync(0)); tdsfs_fetch_wcfst copies the results later. */
typedef struct {            /* caller-owned host SoA, capacity >= tdsfs_candidates_bp / _snp; any member may be NULL */
  int32_t* chrom;           /* as tdsfs_result_t */
  int64_t* start;
  int64_t* end;
  int32_t* snp_count;       /* count_snps, as tdsfs_result_t */
  uint8_t* flags;           /* TDSFS_F_EMPTY */
  int32_t* n_sites;         /* rows that entered the a and b sums */
  double* a;                /* sum of a: variance between populations */
  double* b;                /* sum of b: between individuals within populations */
  double* c;                /* sum of c: between gametes within individuals */
  double* fst;              /* a / ((a + b) + c), NaN when that is 0 */
} tdsfs_wcfst_t;
int tdsfs_wcfst_bp(tdsfs_t* ctx, int64_t W, tdsfs_wcfst_t* out, int64_t cap, int64_t* n_windows);
int tdsfs_wcfst_snp(tdsfs_t* ctx, int64_t N, tdsfs_wcfst_t* out, int64_t cap, int64_t* n_windows);
int tdsfs_fetch_wcfst(tdsfs_t* ctx, tdsfs_wcfst_t* out, int64_t cap, int64_t* n_windows);

/* ---- per-window linkage disequilibrium: Kelly's ZnS and Kim and Nielsen's omega per population (no reference
 * counterpart; DESIGN.md 7) ------------------------------------------------------------------------------------------
 * Same windows and order as tdsfs_diversity_*, for data loaded with tdsfs_load_genotypes only (the counts entry gives
 * TDSFS_ERR_STATE).  Rows: the window's rows that pass the spectrum filter (snp_flags bit0, read directly).  Per population
 * i, samples are its own (not the padding bits of its last pair); dosage and missing calls as in tdsfs_ld_prune (calls held
 * as fix-ups are missing).
 *   site       a row whose called dosages are not all equal (vx > 0 over its own calls).  A row where every called sample
 *              is heterozygous is NOT a site, unlike the segregating sites of tdsfs_neutrality_*;
 *   pair       rows i < j of the window; over the samples called in both, cov, vx, vy as in tdsfs_ld_prune (exact int64).
 *              Defined iff vx vy > 0 (never for a non-site row; two sites can still be undefined through missing calls),
 *              and then r^2 = double(cov^2) / double(vx vy) and q = rint(r^2 2^32) (uint64, round to nearest even);
 *   n_pairs    the defined pairs; zns = 2^-32 double(sum q) / double(n_pairs), each integer converted with round to
 *              nearest; NaN when n_pairs = 0: Kelly's (1997) ZnS over the defined pairs;
 *   omega      with the window's sites s_1 .. s_m in row order, for each split 2 <= k <= m - 2 (L = s_1 .. s_k, R the
 *              rest): WL, WR, X the sums of q over the defined pairs within L, within R and across, nL, nR, nX their
 *              counts, omega_k = (double(WL + WR) / double(nL + nR)) / (double(X) / double(nX)), eligible iff nL + nR > 0
 *              and X > 0.  omega is the largest eligible omega_k (the lowest k on ties), NaN when none is (m < 4
 *              included).  Without missing calls this is Kim and Nielsen's (2004) omega; parity with OmegaPlus is not
 *              claimed (no distance cap, no sub-window grid);
 *   omega_pos  the position of s_k at the best split (the split lies between it and the next site); -1 when omega is NaN.
 * Every sum is an exact integer (window sums in 128 bits), so results are bitwise the same run to run and for any sharding
 * that keeps windows whole.  Cost grows with the square of a window's rows.  Own window arrays, results and per-row
 * scratch (about 49 bytes a loaded row, kept until the handle is destroyed), as tdsfs_diversity_*: a pending plan, the
 * scan's results, the step graph, the other passes' results and tdsfs_ld_prune's buffers are left as they were.
 * out == NULL: enqueue only (honours tdsfs_set_sync(0)); tdsfs_fetch_ld_windows copies the results later. */
typedef struct {            /* caller-owned host SoA, capacity >= tdsfs_candidates_bp / _snp; any member may be NULL */
  int32_t* chrom;           /* as tdsfs_result_t */
  int64_t* start;
  int64_t* end;
  int32_t* snp_count;       /* count_snps, as tdsfs_result_t */
  uint8_t* flags;           /* TDSFS_F_EMPTY */
  int32_t* n_sites_p1;      /* sites m of population 1 */
  int32_t* n_sites_p2;
  int64_t* n_pairs_p1;      /* defined pairs */
  int64_t* n_pairs_p2;
  double* zns_p1;           /* NaN when n_pairs = 0 */
  double* zns_p2;
  double* omega_p1;         /* NaN when no split is eligible */
  double* omega_p2;
  int64_t* omega_pos_p1;    /* position of the last site left of the best split; -1 when omega is NaN */
  int64_t* omega_pos_p2;
} tdsfs_ld_windows_t;
int tdsfs_ld_windows_bp(tdsfs_t* ctx, int64_t W, tdsfs_ld_windows_t* out, int64_t cap, int64_t* n_windows);
int tdsfs_ld_windows_snp(tdsfs_t* ctx, int64_t N, tdsfs_ld_windows_t* out, int64_t cap, int64_t* n_windows);
int tdsfs_fetch_ld_windows(tdsfs_t* ctx, tdsfs_ld_windows_t* out, int64_t cap, int64_t* n_windows);

/* ---- LD pruning of the genotype rows (no reference counterpart; DESIGN.md 7) -----------------------------------------
 * scikit-allel's locate_unlinked (the windowed greedy r^2 rule of PLINK's --indep-pairwise) over the rows loaded with
 * tdsfs_load_genotypes.  Samples: both populations pooled (ns1 + ns2, the padding bits of a population's last pair are not
 * samples).  Dosage: codes 00, 01, 11 give g = 0, 1, 2; code 10 is missing, and so are the calls held as fix-ups (half
 * calls, haploid calls, multi-allelic digits are 10 in the matrix).  r^2 of rows i and j over the n samples called in both,
 * Sx = sum g_i, Sy = sum g_j, Qx = sum g_i^2, Qy = sum g_j^2, P = sum g_i g_j:
 *   cov = n P - Sx Sy,  vx = n Qx - Sx^2,  vy = n Qy - Sy^2   (exact int64),
 *   r^2 = double(cov^2) / double(vx vy)                        (each uint64 converted with round to nearest, one division);
 * undefined, and never pruning, when vx vy = 0 (n = 0 included).  With ns1, ns2 <= 32767 every term is exact.
 * Per chromosome, over rows in loaded order, c0 the chromosome's first row: window k covers rows [c0 + k step,
 * c0 + k step + size) clipped to the chromosome; rows i < j are tested iff a window holds both, j - c0 < floor((i - c0) /
 * step) step + size.  Rows are decided in increasing order: row j is kept iff no kept row i < j tested with j has r^2 >
 * threshold.  This is the final loc of locate_unlinked(gn, size, step, threshold) run on one chromosome in one block
 * (gn = g.to_n_alt(fill=-1)), up to its float32 rounding of r^2.  Parity with PLINK is not claimed.
 * 2 <= size <= 1024, step >= 1 (step > size leaves some neighbouring pairs untested, as in scikit-allel), threshold finite
 * in [0, 1]; else TDSFS_ERR_ARG, as for a NULL keep.  TDSFS_ERR_STATE when nothing is loaded or the counts entry is (it has
 * no calls).  Synchronous: keep (caller-owned host buffer of S bytes) receives 1 for a kept row, 0 for a pruned one, and
 * *n_kept (may be NULL) the kept count.  Own workspace: a pending plan, the scan's unfetched results, the step graph and
 * the per-window passes' results are left as they were. */
int tdsfs_ld_prune(tdsfs_t* ctx, int32_t size, int32_t step, double threshold, uint8_t* keep, int64_t* n_kept);

/* ---- likelihood of explicit spectra ------------------------------------------------------------------------
 * calculate_likelihood_1D / _2D (:478-537, :625-684) on already-interior vectors: x[n] integer counts,
 * b[n] background values, B = sum of b as the caller's language sums it.  *flag = 1 when the reference returns
 * None (sum x == 0 or B == 0). */
int tdsfs_likelihood(tdsfs_t* ctx, const int64_t* x, const double* b, int64_t n, double B, double* T, int32_t* flag);

/* Legacy Poisson composite score, calculate_p (:249-289, twoDSFS.py:336-374): sum over bins with mu != 0 of
 * poisson.logpmf(x, mu), mu = S_w * p_bg. */
int tdsfs_poisson_score(tdsfs_t* ctx, const int64_t* x, const double* mu, int64_t n, double* score);

/* ---- synthetic input (benchmark configs of BASELINE.json) + instrumentation ---------------------------------- */
/* Fill a DEVICE genotype matrix with the synthetic panel of SURVEY.md 8(d): per-SNP ancestral frequency
 * log-uniform, per-population drift, Binomial(2,p) calls, iid missing.  snp0 = global index of row 0. */
int tdsfs_synth_genotypes(tdsfs_t* ctx, void* G_dev, int64_t S, int64_t snp0, int32_t words1, int32_t words2,
                          int32_t ns1, int32_t ns2, uint64_t seed, double missing_rate, double fst);
/* CUDA-event times (ms) of the last background / finalize / scan calls (synchronises the stream):
 * [0]=count kernel (K1), [1]=finalize, [2]=boundaries (K2), [3]=score small windows (K3/K4), [4]=score large windows,
 * [5]=background call, [6]=scan call, [7]=K1 start -> last score kernel end, [8]=peer exchange kernel (n >= 9),
 * [9]=segment + finish kernels of the last tdsfs_diversity_* call (n >= 10),
 * [10]=segment + finish kernels of the last tdsfs_neutrality_* call (n >= 11),
 * [11]=segment + finish kernels of the last tdsfs_wcfst_* call (n >= 12),
 * [12]=k_ld_pairs and [13]=k_ld_resolve of the last tdsfs_ld_prune call (n >= 14),
 * [14]=pair + finish kernels of the last tdsfs_ld_windows_* call (n >= 15). */
int tdsfs_timings(tdsfs_t* ctx, float* ms, int32_t n);
int64_t tdsfs_launch_count(tdsfs_t* ctx); /* kernels launched by this handle so far */
/* Which path scored the last scan: *fused = 1 when the fused pair ran (tdsfs_plan_* before tdsfs_background on the
 * genotype-level entry: the count kernel leaves every window's background-independent sums and one finish kernel gathers
 * ln b over the per-SNP records), 0 for the table scorer; *record_bytes = 4 (narrow per-SNP record) or 8. */
int tdsfs_scan_info(tdsfs_t* ctx, int32_t* fused, int32_t* record_bytes);
/* Diagnostics (handles created with TDSFS_TAIL_STAMPS=1 in the environment, else TDSFS_ERR_STATE): SM clock (clock64) of
 * CTA 0 of the last count kernel that ran a tail: [0] kernel entry, [1] its histograms flushed, [2] past the grid barrier,
 * [3] past the first peer barrier, [4] its slice pushed and fenced, [5] past the second peer barrier, [6] ln tables written,
 * [7] totals written.  No reference counterpart. */
int tdsfs_tail_stamps(tdsfs_t* ctx, uint64_t* out8);
int tdsfs_version(void);

#ifdef __cplusplus
}
#endif
#endif /* TDSFS_H */
