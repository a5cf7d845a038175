// tdsfs_diversity.cuh -- per-window Hudson FST, pi and dxy, per-population Watterson's theta and Tajima's D, and Weir and
// Cockerham's FST (DESIGN.md section 7).  Included by tdsfs.cu after tdsfs_kernels.cuh and tdsfs_fused.cuh.  No reference
// counterpart: the reference's users get the FST column of their tables from pixy, and Tajima's D from scikit-allel, run
// separately over the same VCF.
//
// Per SNP that passes the spectrum filters (snp_flags bit0) with n_i = ref_i + alt_i >= 2 in both populations, in fp64:
//   pi_i = 2 ref_i alt_i / (n_i (n_i - 1)),   dxy = (ref_1 alt_2 + alt_1 ref_2) / (n_1 n_2)
// (integer numerators and denominators, one rounded division each).  The sums of a window are taken in a fixed order that
// depends on the window's rows alone: segments of DIV_SEG rows counted from the window's first row; inside a segment lane
// (s - first row) mod 32 adds its SNPs in row order and a fixed xor tree combines the lanes; the segment sums are added in
// segment order.  So the result is bitwise the same for the counts and the genotype entry, any grid and any sharding that
// keeps windows whole.
#pragma once

namespace tdsfs {

constexpr int DIV_SEG = 1024;   // rows per segment (a multiple of 32)
constexpr int DIV_WARPS = 8;    // warps per CTA of k_diversity, k_neutrality and k_wcfst: one warp per segment

// The segment list of a pass's candidate windows: window w owns segments [segoff[w], segoff[w + 1]), DIV_SEG rows each
// counted from its first row (the last one shorter).
struct SegList {
  const int32_t* wlo;          // [ncand] first row of each candidate window (k2_bounds_*)
  const int32_t* whi;          // [ncand] one past its last row
  long long ncand;
  const long long* segoff;     // [ncand + 1] exclusive prefix sum of k_div_nseg's counts: segoff[ncand] = number of segments
};

// Segments per window, 0 in the last slot [ncand]: the exclusive scan of nseg is the segment list's segoff.
__global__ void __launch_bounds__(256) k_div_nseg(const int32_t* wlo, const int32_t* whi, long long ncand, long long* nseg) {
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id < ncand) nseg[id] = (__ldg(whi + id) - __ldg(wlo + id) + DIV_SEG - 1) / DIV_SEG;
  else if (id == ncand) nseg[id] = 0;
}

// (ref1, alt1, ref2, alt2) of SNP s before the fix-ups and its heterozygous calls (het1, het2): compile-time word counts
// (fully unrolled, every load of the row issued together) or the runtime decode shared with k_window_hist (any width, and
// the counts entry, whose het counts are 0).  A pass that does not read het1 / het2 compiles to the same code without them.
template <int TW1, int TW2>
__device__ __forceinline__ void div_counts(const KeyParams& p, long long s, int& ref1, int& alt1, int& ref2, int& alt2,
                                           int& het1, int& het2) {
  if constexpr (TW1 > 0 && TW2 > 0) {
    // every word of the row is loaded before any is counted: one memory round trip per row (count_pop_planes interleaves
    // loads and counting, and the compiler then issues the second population's loads only after the first one's arrive)
    constexpr int P1 = TW1 / 2, P2 = TW2 / 2;
    const uint32_t* row = p.G + (s >> 5) * (long long)((TW1 + TW2) * BLK) + (s & 31);
    uint32_t lo1[P1], hi1[P1], lo2[P2], hi2[P2];
#pragma unroll
    for (int i = 0; i < P1; ++i) { lo1[i] = __ldcs(row + (2 * i) * BLK); hi1[i] = __ldcs(row + (2 * i + 1) * BLK); }
#pragma unroll
    for (int i = 0; i < P2; ++i) { lo2[i] = __ldcs(row + (TW1 + 2 * i) * BLK); hi2[i] = __ldcs(row + (TW1 + 2 * i + 1) * BLK); }
    // codes 00, 01, 11, 10 = hom-ref, het, hom-alt, missing: alt = popc(lo) + popc(lo & hi), missing = popc(hi) - popc(lo & hi),
    // het = popc(lo & ~hi) = popc(lo) - popc(lo & hi) = alt - 2 popc(lo & hi)
    uint32_t b1[P1], b2[P2];
#pragma unroll
    for (int i = 0; i < P1; ++i) b1[i] = lo1[i] & hi1[i];
#pragma unroll
    for (int i = 0; i < P2; ++i) b2[i] = lo2[i] & hi2[i];
    const int c1 = (int)popc_sum<P1>(b1), c2 = (int)popc_sum<P2>(b2);
    alt1 = (int)popc_sum<P1>(lo1) + c1;
    alt2 = (int)popc_sum<P2>(lo2) + c2;
    ref1 = 2 * (p.ns1 - ((int)popc_sum<P1>(hi1) - c1)) - alt1;
    ref2 = 2 * (p.ns2 - ((int)popc_sum<P2>(hi2) - c2)) - alt2;
    het1 = alt1 - 2 * c1;
    het2 = alt2 - 2 * c2;
  } else {
    source_counts(p, s, ref1, alt1, ref2, alt2, het1, het2);
  }
}

// Rows [r0, r1) of segment g: segment g - segoff[w] of window w, the last w with segoff[w] <= g (an empty window owns no
// segment, so it is never the last one).  False for a warp past the last segment: the grid covers a bound on their number.
__device__ __forceinline__ bool segment_rows(const SegList& seg, long long g, long long& r0, long long& r1) {
  if (g >= __ldg(seg.segoff + seg.ncand)) return false;
  long long lo = 0, hi = seg.ncand;
  while (hi - lo > 1) {
    const long long mid = (lo + hi) >> 1;
    if (__ldg(seg.segoff + mid) <= g) lo = mid; else hi = mid;
  }
  r0 = (long long)__ldg(seg.wlo + lo) + (g - __ldg(seg.segoff + lo)) * DIV_SEG;
  r1 = min(r0 + DIV_SEG, (long long)__ldg(seg.whi + lo));
  return true;
}

// The NF fp sums of the segment [r0, r1), taken by one warp in the order that defines them (top of this file).  The warp
// walks the ALIGNED 32-row blocks that overlap its segment, so word w of a step is exactly one 128-byte line (a window
// starting inside a block would otherwise split every line of every step in two).  Lane l loads row s = b + l, and
// row(s, ref1, alt1, ref2, alt2, het1, het2, t) sets that row's terms t[] and adds the pass's integer statistics to the
// lane's own registers: integers, so the kernel reduces them over the warp at the end in any order.  The terms move to
// the lane that owns row s in the definition, (s - r0) mod 32 = (l - r0) mod 32, which receives its rows in increasing
// order, one per block, and a fixed xor tree combines the lanes: the sums are the definition's, bit for bit.
//
// Every lane adds a term in every block, +0.0 for a row outside the segment or one that adds no term.  That leaves a sum
// bitwise unchanged as long as no term is -0.0: every sum starts at +0.0, and under round-to-nearest a sum of operands
// none of which is -0.0 is never -0.0 (an exact zero sum of operands of opposite signs is +0.0), while x + (+0.0) is x bit
// for bit for any x but -0.0.  Terms may be negative.  Each pass's terms are an integer numerator over a nonzero integer
// denominator, converted and divided with round-to-nearest: a zero numerator gives +0.0 and a nonzero one a quotient far
// above the underflow range, so no term is ever -0.0.
template <int TW1, int TW2, int NF, typename Row>
__device__ __forceinline__ void segment_sums(const KeyParams& k, long long r0, long long r1, double (&sum)[NF], Row row) {
  const int lane = threadIdx.x & 31;
  const int src = (lane + (int)(r0 & 31)) & 31;  // the lane that loads the row this lane owns
#pragma unroll
  for (int i = 0; i < NF; ++i) sum[i] = 0.0;
  for (long long b = r0 & ~31LL; b < r1; b += 32) {
    const long long s = b + lane;
    double t[NF];
#pragma unroll
    for (int i = 0; i < NF; ++i) t[i] = 0.0;
    if (s >= r0 && s < r1) {
      int ref1, alt1, ref2, alt2, het1, het2;
      div_counts<TW1, TW2>(k, s, ref1, alt1, ref2, alt2, het1, het2);
      row(s, ref1, alt1, ref2, alt2, het1, het2, t);
    }
#pragma unroll
    for (int i = 0; i < NF; ++i) sum[i] += __shfl_sync(0xffffffffu, t[i], src);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
#pragma unroll
    for (int i = 0; i < NF; ++i) sum[i] += __shfl_xor_sync(0xffffffffu, sum[i], o);
  }
}

// ------------------------------------------------------------------------------------------------ Hudson FST, pi, dxy
struct DivPart {  // sums of one segment
  double pi1, pi2, dxy;
  int n_sites, snp_count;
};

struct DivParams {
  KeyParams k;                 // source rows (G or cnt), sample columns, snp_flags + fix-ups (row_filters)
  SegList seg;
  DivPart* part;               // [segments]
  int32_t* snp_count;          // [ncand] outputs
  int32_t* n_sites;
  double* pi1;
  double* pi2;
  double* dxy;
  double* fst;
  uint8_t* flags;
};

// One warp per segment: its pi_1, pi_2 and dxy sums, SNPs that entered them and SNPs counted.
template <int TW1, int TW2>
__global__ void __launch_bounds__(DIV_WARPS * 32) k_diversity(const __grid_constant__ DivParams p) {
  const long long g = (long long)blockIdx.x * DIV_WARPS + (threadIdx.x >> 5);
  long long r0, r1;
  if (!segment_rows(p.seg, g, r0, r1)) return;
  double sum[3];  // pi1, pi2, dxy
  int n_sites = 0, snp_count = 0;
  segment_sums<TW1, TW2>(p.k, r0, r1, sum, [&](long long s, int ref1, int alt1, int ref2, int alt2, int, int, double (&t)[3]) {
    snp_count += p.k.flags ? (__ldg(p.k.flags + s) >> 1) & 1 : 1;
    const bool pass = row_filters(p.k, s, ref1, alt1, ref2, alt2);
    const long long n1 = ref1 + alt1, n2 = ref2 + alt2;
    if (pass && n1 >= 2 && n2 >= 2) {
      t[0] = (double)(2LL * ref1 * alt1) / (double)(n1 * (n1 - 1));
      t[1] = (double)(2LL * ref2 * alt2) / (double)(n2 * (n2 - 1));
      t[2] = (double)((long long)ref1 * alt2 + (long long)alt1 * ref2) / (double)(n1 * n2);
      ++n_sites;
    }
  });
  n_sites = __reduce_add_sync(0xffffffffu, n_sites);
  snp_count = __reduce_add_sync(0xffffffffu, snp_count);
  if ((threadIdx.x & 31) == 0) p.part[g] = DivPart{sum[0], sum[1], sum[2], n_sites, snp_count};
}

// One thread per window: its segment sums in segment order, then FST (NaN when dxy == 0).
__global__ void __launch_bounds__(256) k_div_finish(const __grid_constant__ DivParams p) {
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= p.seg.ncand) return;
  double pi1 = 0.0, pi2 = 0.0, dxy = 0.0;
  int n_sites = 0, snp_count = 0;
  for (long long g = __ldg(p.seg.segoff + id), e = __ldg(p.seg.segoff + id + 1); g < e; ++g) {
    const DivPart q = p.part[g];
    pi1 += q.pi1; pi2 += q.pi2; dxy += q.dxy;
    n_sites += q.n_sites; snp_count += q.snp_count;
  }
  p.snp_count[id] = snp_count;
  p.n_sites[id] = n_sites;
  p.pi1[id] = pi1;
  p.pi2[id] = pi2;
  p.dxy[id] = dxy;
  p.fst[id] = dxy == 0.0 ? __longlong_as_double(0x7FF8000000000000LL) : 1.0 - (pi1 + pi2) / (2.0 * dxy);
  p.flags[id] = __ldg(p.seg.whi + id) == __ldg(p.seg.wlo + id) ? TDSFS_F_EMPTY : 0;
}

// ------------------------------------------------------------------------------------------------ neutrality
// Per population i, over the rows that pass the spectrum filters: S_i segregating sites (ref_i > 0 and alt_i > 0),
// n_max_i the largest n_i, theta_pi_i the sum of 2 ref_i alt_i / (n_i (n_i - 1)) over the rows with n_i >= 2 (the pi_i term
// of the FST pass, summed in the same order, but not restricted to rows where the other population has n >= 2); then
// Watterson's theta S_i / a1(n_max_i) and Tajima's D (Tajima 1989) at n = n_max_i.  A window's results depend on its rows
// alone, as the FST pass's do.

struct NeutPart {  // sums of one segment
  double theta_pi1, theta_pi2;
  int S1, S2, nmax1, nmax2, snp_count;
};

struct NeutParams {
  KeyParams k;                 // source rows, sample columns, snp_flags + fix-ups
  SegList seg;
  NeutPart* part;              // [segments]
  const double* a1;            // [tab_n + 1] a1(n) = sum_{k=1}^{n-1} 1/k, ascending k; a1(0) = a1(1) = 0
  const double* a2;            // [tab_n + 1] a2(n) = sum_{k=1}^{n-1} 1/k^2
  int32_t* snp_count;          // [ncand] outputs
  int32_t* S1;
  int32_t* S2;
  int32_t* nmax1;
  int32_t* nmax2;
  double* theta_pi1;
  double* theta_pi2;
  double* theta_w1;
  double* theta_w2;
  double* tajd1;
  double* tajd2;
  uint8_t* flags;
};

// One warp per segment: its theta_pi sums, segregating sites, largest n and SNPs counted, per population.
template <int TW1, int TW2>
__global__ void __launch_bounds__(DIV_WARPS * 32) k_neutrality(const __grid_constant__ NeutParams p) {
  const long long g = (long long)blockIdx.x * DIV_WARPS + (threadIdx.x >> 5);
  long long r0, r1;
  if (!segment_rows(p.seg, g, r0, r1)) return;
  double sum[2];  // theta_pi1, theta_pi2
  int S1 = 0, S2 = 0, nmax1 = 0, nmax2 = 0, snp_count = 0;
  segment_sums<TW1, TW2>(p.k, r0, r1, sum, [&](long long s, int ref1, int alt1, int ref2, int alt2, int, int, double (&t)[2]) {
    snp_count += p.k.flags ? (__ldg(p.k.flags + s) >> 1) & 1 : 1;
    if (row_filters(p.k, s, ref1, alt1, ref2, alt2)) {
      const long long n1 = ref1 + alt1, n2 = ref2 + alt2;
      S1 += ref1 > 0 && alt1 > 0;
      S2 += ref2 > 0 && alt2 > 0;
      nmax1 = max(nmax1, (int)n1);
      nmax2 = max(nmax2, (int)n2);
      if (n1 >= 2) t[0] = (double)(2LL * ref1 * alt1) / (double)(n1 * (n1 - 1));
      if (n2 >= 2) t[1] = (double)(2LL * ref2 * alt2) / (double)(n2 * (n2 - 1));
    }
  });
  S1 = __reduce_add_sync(0xffffffffu, S1);
  S2 = __reduce_add_sync(0xffffffffu, S2);
  snp_count = __reduce_add_sync(0xffffffffu, snp_count);
  nmax1 = __reduce_max_sync(0xffffffffu, nmax1);
  nmax2 = __reduce_max_sync(0xffffffffu, nmax2);
  if ((threadIdx.x & 31) == 0) p.part[g] = NeutPart{sum[0], sum[1], S1, S2, nmax1, nmax2, snp_count};
}

// Watterson's theta and Tajima's D of one population from (theta_pi, S, n_max); NaN where undefined.
__device__ __forceinline__ void tajima(const NeutParams& p, double pi, int S, int n, double& theta_w, double& d) {
  const double nan = __longlong_as_double(0x7FF8000000000000LL);
  theta_w = nan;
  d = nan;
  if (n < 2) return;
  const double a1 = __ldg(p.a1 + n), a2 = __ldg(p.a2 + n), nn = n, s = S;
  theta_w = s / a1;
  if (S < 3) return;
  const double b1 = (nn + 1.0) / (3.0 * (nn - 1.0));
  const double b2 = 2.0 * (nn * nn + nn + 3.0) / (9.0 * nn * (nn - 1.0));
  const double c1 = b1 - 1.0 / a1;
  const double c2 = b2 - (nn + 2.0) / (a1 * nn) + a2 / (a1 * a1);
  const double e1 = c1 / a1, e2 = c2 / (a1 * a1 + a2);
  const double var = e1 * s + e2 * s * (s - 1.0);
  if (var > 0.0) d = (pi - theta_w) / sqrt(var);
}

// One thread per window: its segment parts in segment order (maxima for n_max), then theta_W and Tajima's D.
__global__ void __launch_bounds__(256) k_neut_finish(const __grid_constant__ NeutParams p) {
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= p.seg.ncand) return;
  double pi1 = 0.0, pi2 = 0.0;
  int S1 = 0, S2 = 0, nmax1 = 0, nmax2 = 0, snp_count = 0;
  for (long long g = __ldg(p.seg.segoff + id), e = __ldg(p.seg.segoff + id + 1); g < e; ++g) {
    const NeutPart q = p.part[g];
    pi1 += q.theta_pi1; pi2 += q.theta_pi2;
    S1 += q.S1; S2 += q.S2; snp_count += q.snp_count;
    nmax1 = max(nmax1, q.nmax1); nmax2 = max(nmax2, q.nmax2);
  }
  double tw1, tw2, d1, d2;
  tajima(p, pi1, S1, nmax1, tw1, d1);
  tajima(p, pi2, S2, nmax2, tw2, d2);
  p.snp_count[id] = snp_count;
  p.S1[id] = S1; p.S2[id] = S2;
  p.nmax1[id] = nmax1; p.nmax2[id] = nmax2;
  p.theta_pi1[id] = pi1; p.theta_pi2[id] = pi2;
  p.theta_w1[id] = tw1; p.theta_w2[id] = tw2;
  p.tajd1[id] = d1; p.tajd2[id] = d2;
  p.flags[id] = __ldg(p.seg.whi + id) == __ldg(p.seg.wlo + id) ? TDSFS_F_EMPTY : 0;
}

// ------------------------------------------------------------------------------------------------ Weir and Cockerham's FST
// Per row that passes the spectrum filter (snp_flags bit0, read directly: no fix-up is applied, so the calls held as
// fix-ups count as missing), from the 2-bit codes of population i: n_i called diploids, x_i their alt alleles, h_i their
// heterozygotes; N = n1 + n2, X = x1 + x2, H = h1 + h2, D = x1 n2 - x2 n1.  The variance components summed over both
// alleles (scikit-allel's weir_cockerham_fst with r = 2), each an exact int64 numerator over an exact int64 denominator
// with one rounded division:
//   a = [D^2 (N-1) - n1 n2 (X(2N-X) - N H)] / [4 n1^2 n2^2 (N-2)]   rows with n1 >= 1, n2 >= 1 and N >= 3 (n_sites)
//   b = [n1 n2 (X(2N-X) - 2(N-1) H) - D^2] / [2 n1 n2 N (N-2)]      the same rows
//   c = H / N                                                     rows with N >= 1
// Every numerator and denominator stays below 2^63 while ns1, ns2 <= WC_MAX_SAMPLES (the largest, 4 n1^2 n2^2 (N-1) and
// 4 n1^2 n2^2 (N-2), are about 8.19e18 at 4000 + 4000).  The window sums run in the order of the FST pass, and
// fst = a / ((a + b) + c), NaN when that denominator is 0.
constexpr int WC_MAX_SAMPLES = 4000;

struct WcPart {  // sums of one segment
  double a, b, c;
  int n_sites, snp_count;
};

struct WcParams {
  KeyParams k;                 // genotype rows, sample columns, snp_flags
  SegList seg;
  WcPart* part;                // [segments]
  int32_t* snp_count;          // [ncand] outputs
  int32_t* n_sites;
  double* a;
  double* b;
  double* c;
  double* fst;
  uint8_t* flags;
};

// One warp per segment: its a, b and c sums, rows that entered a and b, and SNPs counted.
template <int TW1, int TW2>
__global__ void __launch_bounds__(DIV_WARPS * 32) k_wcfst(const __grid_constant__ WcParams p) {
  const long long g = (long long)blockIdx.x * DIV_WARPS + (threadIdx.x >> 5);
  long long r0, r1;
  if (!segment_rows(p.seg, g, r0, r1)) return;
  double sum[3];  // a, b, c
  int n_sites = 0, snp_count = 0;
  segment_sums<TW1, TW2>(p.k, r0, r1, sum, [&](long long s, int ref1, int alt1, int ref2, int alt2, int het1, int het2,
                                               double (&t)[3]) {
    const int f = p.k.flags ? __ldg(p.k.flags + s) : 3;
    snp_count += (f >> 1) & 1;
    const int n1 = (ref1 + alt1) >> 1, n2 = (ref2 + alt2) >> 1, N = n1 + n2;  // ref + alt = 2 (ns - missing)
    if (!(f & 1) || N < 1) return;
    const int X = alt1 + alt2, H = het1 + het2;
    t[2] = (double)H / (double)N;
    if (n1 < 1 || n2 < 1 || N < 3) return;
    // With ns1, ns2 <= WC_MAX_SAMPLES every factor fits in 32 bits (|D| <= 2 n1 n2, X(2N-X) <= N^2, 2(N-1)H < 2N^2), so
    // each product is one 32 x 32 -> 64-bit multiply, and at most one more by a 32-bit factor
    const int D = alt1 * n2 - alt2 * n1, n12 = n1 * n2, Q = X * (2 * N - X);
    const long long D2 = (long long)D * D;
    t[0] = (double)(D2 * (N - 1) - (long long)n12 * (Q - N * H)) / (double)((long long)n12 * n12 * (4 * (N - 2)));
    t[1] = (double)((long long)n12 * (Q - 2 * (N - 1) * H) - D2) / (double)((long long)n12 * N * (2 * (N - 2)));
    ++n_sites;
  });
  n_sites = __reduce_add_sync(0xffffffffu, n_sites);
  snp_count = __reduce_add_sync(0xffffffffu, snp_count);
  if ((threadIdx.x & 31) == 0) p.part[g] = WcPart{sum[0], sum[1], sum[2], n_sites, snp_count};
}

// One thread per window: its segment sums in segment order, then fst = a / ((a + b) + c) (NaN when that is 0).
__global__ void __launch_bounds__(256) k_wc_finish(const __grid_constant__ WcParams p) {
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= p.seg.ncand) return;
  double a = 0.0, b = 0.0, c = 0.0;
  int n_sites = 0, snp_count = 0;
  for (long long g = __ldg(p.seg.segoff + id), e = __ldg(p.seg.segoff + id + 1); g < e; ++g) {
    const WcPart q = p.part[g];
    a += q.a; b += q.b; c += q.c;
    n_sites += q.n_sites; snp_count += q.snp_count;
  }
  const double den = (a + b) + c;
  p.snp_count[id] = snp_count;
  p.n_sites[id] = n_sites;
  p.a[id] = a;
  p.b[id] = b;
  p.c[id] = c;
  p.fst[id] = den == 0.0 ? __longlong_as_double(0x7FF8000000000000LL) : a / den;
  p.flags[id] = __ldg(p.seg.whi + id) == __ldg(p.seg.wlo + id) ? TDSFS_F_EMPTY : 0;
}

}  // namespace tdsfs
