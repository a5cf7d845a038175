// tdsfs_ld.cuh -- LD pruning of the loaded genotype rows (DESIGN.md section 7): scikit-allel's locate_unlinked, the
// windowed greedy r^2 rule of PLINK's --indep-pairwise.  Included by tdsfs.cu after tdsfs_kernels.cuh.
//
// Samples are those of both populations pooled; codes 00, 01, 11 give dosage g = 0, 1, 2 and code 10 is missing (calls
// held as fix-ups are 10 in the matrix, so they count as missing); the padding bits of a population's last (lo, hi) pair
// are not samples.  r^2 of rows i and j over the n samples called in both, from exact integer sums:
//   cov = n P - Sx Sy,  vx = n Qx - Sx^2,  vy = n Qy - Sy^2,  r^2 = double(cov^2) / double(vx vy)   (undefined when vx vy = 0)
// With ns1, ns2 <= 32767, n <= 65534 and cov^2 <= vx vy <= n^4 < 2^64: every term is exact in (u)int64.
// Per chromosome, rows i < j are tested iff a window [c0 + k step, c0 + k step + size) holds both, and row j is kept iff no
// kept row i < j tested with j has r^2 > threshold.
#pragma once

namespace tdsfs {

constexpr int LD_MAX_SIZE = 1024;          // window rows: the kept bits of the last 1023 rows are one register per lane of a warp
constexpr int LD_WARPS = 8;                // warps per CTA of k_ld_pairs
constexpr int LD_IROWS = BLK / LD_WARPS;   // rows i per warp of one 32-row i block
constexpr int LD_KP = 32;                  // (lo, hi) word pairs of both populations staged at a time

struct LdParams {
  const uint32_t* G;           // B32 genotype matrix
  long long S;
  int W1, W2, ns1, ns2;
  const long long* chrom_off;  // [C + 1]
  int C;
  int size, step, mw;          // window rows, window step, mask words per row = ceil((size - 1) / 32)
  double thr;
  uint32_t* mask;              // [S * mw] bit d - 1 of row j: rows j - d and j are tested and their r^2 > thr
  uint8_t* keep;               // [S] 1 = kept
  unsigned long long* n_kept;
};

// First row of the chromosome that holds row s (empty chromosomes are skipped: off[lo] <= s < off[lo + 1]).
__device__ __forceinline__ long long ld_chrom_start(const LdParams& p, long long s) {
  int lo = 0, hi = p.C;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(p.chrom_off + mid) <= s) lo = mid; else hi = mid;
  }
  return __ldg(p.chrom_off + lo);
}

// Rows i < j of the chromosome that starts at c0 share a window.
__device__ __forceinline__ bool ld_tested(const LdParams& p, long long i, long long j, long long c0) {
  return i >= c0 && i < j && j - c0 < (i - c0) / p.step * (long long)p.step + p.size;
}

// Sample bits of word pair q (population 1's pairs, then population 2's) that are not padding.  P: LdParams or LdwParams.
template <typename P>
__device__ __forceinline__ uint32_t ld_valid(const P& p, int q) {
  const int h1 = p.W1 >> 1;
  const int left = q < h1 ? p.ns1 - 32 * q : p.ns2 - 32 * (q - h1);
  return left >= 32 ? 0xffffffffu : (left <= 0 ? 0u : (1u << left) - 1u);
}

// Planes of one 32-row B32 block's word pair q: called c = (lo | ~hi), d1 = lo (g >= 1), d2 = lo & hi (g = 2).  d1 and d2
// are 0 on missing calls; all three are masked to the pair's samples.
template <typename P>
__device__ __forceinline__ uint3 ld_planes(const P& p, long long blk, int RW, int q, int r) {
  const uint32_t* w = p.G + (blk * RW + 2 * q) * BLK + r;
  const uint32_t lo = __ldg(w), hi = __ldg(w + BLK), v = ld_valid(p, q);
  return make_uint3((lo | ~hi) & v, lo & v, lo & hi & v);
}

// One CTA per 32-row block of rows j: the mask words of its rows.  It streams the 32-row blocks of rows i from the first
// row any of its rows is tested with up to its own block, LD_KP word pairs at a time: the j block's planes in shared memory
// at [(q * 3 + plane) * 32 + row] (lane l reads bank l), the i block's as one 16-byte (c, d1, d2) entry per (q, row) (a
// broadcast to the warp).  Lane l of warp w holds the sums of row j = j0 + l with the LD_IROWS rows i = i0 + w LD_IROWS + k,
// 9 popcounts per word pair each:
//   n += popc(cx & cy),  ax += popc(d1x & cy), bx += popc(d2x & cy)  (Sx = ax + bx, Qx = ax + 3 bx; likewise y),
//   P += popc(d1x & d1y) + popc(d1x & d2y) + popc(d2x & d1y) + popc(d2x & d2y).
// A warp none of whose pairs is tested skips the arithmetic of that i block.
template <int TW1, int TW2>
__global__ void __launch_bounds__(LD_WARPS * 32) k_ld_pairs(const __grid_constant__ LdParams p) {
  constexpr int TNP = (TW1 + TW2) / 2;  // word pairs per row; 0: runtime
  __shared__ uint32_t sj[LD_KP * 3 * BLK];
  __shared__ uint4 si[LD_KP * BLK];
  __shared__ uint32_t sm[BLK * (LD_MAX_SIZE / 32)];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int NP = TNP > 0 ? TNP : (p.W1 + p.W2) >> 1, RW = 2 * NP;
  const int nch = (NP + LD_KP - 1) / LD_KP;
  const long long jb = blockIdx.x, j0 = jb * BLK, j = j0 + lane;
  const bool jok = j < p.S;
  const long long c0 = ld_chrom_start(p, jok ? j : p.S - 1);
  const long long first = max(ld_chrom_start(p, j0), j0 - p.size + 1);
  for (int t = threadIdx.x; t < BLK * p.mw; t += blockDim.x) sm[t] = 0u;

  auto stage_j = [&](int q0, int nq) {
    for (int t = threadIdx.x; t < nq * BLK; t += blockDim.x) {
      const int q = t >> 5, r = t & 31;
      const uint3 v = ld_planes(p, jb, RW, q0 + q, r);
      sj[(q * 3 + 0) * BLK + r] = v.x;
      sj[(q * 3 + 1) * BLK + r] = v.y;
      sj[(q * 3 + 2) * BLK + r] = v.z;
    }
  };
  if (nch == 1) stage_j(0, NP);

  for (long long ib = first >> 5; ib <= jb; ++ib) {
    const long long i0 = ib * BLK + warp * LD_IROWS;
    bool any = false;
#pragma unroll
    for (int k = 0; k < LD_IROWS; ++k) any |= jok && ld_tested(p, i0 + k, j, c0);
    any = __any_sync(0xffffffffu, any);
    int n[LD_IROWS], ax[LD_IROWS], bx[LD_IROWS], ay[LD_IROWS], by[LD_IROWS], pp[LD_IROWS];
#pragma unroll
    for (int k = 0; k < LD_IROWS; ++k) n[k] = ax[k] = bx[k] = ay[k] = by[k] = pp[k] = 0;
    for (int ch = 0; ch < nch; ++ch) {
      const int q0 = ch * LD_KP, nq = TNP > 0 ? TNP : min(LD_KP, NP - q0);
      __syncthreads();  // the previous pass's readers of sj / si are done
      if (nch > 1) stage_j(q0, nq);
      for (int t = threadIdx.x; t < nq * BLK; t += blockDim.x) {
        const int q = t >> 5, r = t & 31;
        const uint3 v = ld_planes(p, ib, RW, q0 + q, r);
        si[q * BLK + r] = make_uint4(v.x, v.y, v.z, 0u);
      }
      __syncthreads();
      if (!any) continue;
#pragma unroll 4
      for (int q = 0; q < nq; ++q) {
        const uint32_t cy = sj[(q * 3 + 0) * BLK + lane], d1y = sj[(q * 3 + 1) * BLK + lane], d2y = sj[(q * 3 + 2) * BLK + lane];
#pragma unroll
        for (int k = 0; k < LD_IROWS; ++k) {
          const uint4 x = si[q * BLK + warp * LD_IROWS + k];
          n[k] += __popc(x.x & cy);
          ax[k] += __popc(x.y & cy);
          bx[k] += __popc(x.z & cy);
          ay[k] += __popc(d1y & x.x);
          by[k] += __popc(d2y & x.x);
          pp[k] += __popc(x.y & d1y) + __popc(x.y & d2y) + __popc(x.z & d1y) + __popc(x.z & d2y);
        }
      }
    }
    if (!any) continue;
#pragma unroll
    for (int k = 0; k < LD_IROWS; ++k) {
      const long long i = i0 + k;
      if (!jok || !ld_tested(p, i, j, c0)) continue;
      const long long nn = n[k], sx = ax[k] + bx[k], sy = ay[k] + by[k];
      const long long cov = nn * pp[k] - sx * sy;
      const unsigned long long vx = (unsigned long long)(nn * (ax[k] + 3LL * bx[k]) - sx * sx);
      const unsigned long long vy = (unsigned long long)(nn * (ay[k] + 3LL * by[k]) - sy * sy);
      const unsigned long long den = vx * vy;
      if (den == 0) continue;  // r^2 undefined: never prunes
      const unsigned long long ac = (unsigned long long)(cov < 0 ? -cov : cov);
      if (__ull2double_rn(ac * ac) / __ull2double_rn(den) > p.thr) {
        const int d = (int)(j - i) - 1;
        atomicOr(&sm[lane * p.mw + (d >> 5)], 1u << (d & 31));
      }
    }
  }
  __syncthreads();
  const long long rows = min((long long)BLK, p.S - j0);
  for (int t = threadIdx.x; t < rows * p.mw; t += blockDim.x) p.mask[j0 * p.mw + t] = sm[t];
}

// The greedy decision: one warp per chromosome, 32 rows (a group, counted from the chromosome's first row) per step.  Lane
// g mod 32 holds the kept bits of group g in one register, for the last 32 groups: the 1023 rows before any row of the
// current group.  Lane l (row j = base + l) aligns, per mask word k, the kept bits of rows j - 32k - 32 .. j - 32k - 1 with
// one funnel shift of two broadcast registers, and ANDs them with the word: any hit prunes the row.  The dependencies
// inside the group (mask word 0, rows base .. j - 1) are resolved in 32 dependent ballots.
__global__ void __launch_bounds__(32) k_ld_resolve(const __grid_constant__ LdParams p) {
  const int lane = threadIdx.x;
  const long long c0 = __ldg(p.chrom_off + blockIdx.x), c1 = __ldg(p.chrom_off + blockIdx.x + 1);
  uint32_t ring = 0u;
  unsigned long long total = 0;
  for (long long t = 0, base = c0; base < c1; ++t, base += BLK) {
    const long long j = base + lane;
    const bool row = j < c1;
    uint32_t m[LD_MAX_SIZE / 32];
#pragma unroll
    for (int k = 0; k < LD_MAX_SIZE / 32; ++k) m[k] = row && k < p.mw ? __ldg(p.mask + j * p.mw + k) : 0u;
    uint32_t hit = 0u;
#pragma unroll
    for (int k = 0; k < LD_MAX_SIZE / 32; ++k) {
      if (k >= p.mw) break;
      const long long g0 = t - k - 1;  // >= t - 32: its slot still holds it while the current group is open
      const uint32_t lo = __shfl_sync(0xffffffffu, ring, (int)(g0 & 31));
      const uint32_t hi = __shfl_sync(0xffffffffu, ring, (int)((g0 + 1) & 31));
      const uint32_t v = __funnelshift_r(g0 >= 0 ? lo : 0u, k > 0 && g0 + 1 >= 0 ? hi : 0u, lane);  // bit q: row j - 32k - 32 + q
      hit |= __brev(v) & m[k];
    }
    const uint32_t below = m[0] & ((1u << lane) - 1u);         // bit d - 1: row j - d of this group
    const uint32_t dep = lane ? __brev(below) >> (32 - lane) : 0u;  // bit s: row base + s
    const bool open = row && hit == 0u;
    uint32_t kept = 0u;
    for (int s = 0; s < 32; ++s) kept |= __ballot_sync(0xffffffffu, open && !(dep & kept)) & (1u << s);
    if (lane == (int)(t & 31)) ring = kept;
    if (row) p.keep[j] = (kept >> lane) & 1u;
    total += __popc(kept);
  }
  if (lane == 0 && total) atomicAdd(p.n_kept, total);
}

// ------------------------------------------------------------------------------------------------ per-window LD
// Kelly's ZnS and Kim and Nielsen's omega per candidate window and population (DESIGN.md section 7).  Rows are the window's
// rows that pass the spectrum filter (snp_flags bit0, read directly: calls held as fix-ups are missing, as above).  Per
// population, over its own samples: a row is a site iff its called dosages are not all equal (vx > 0 over its own calls);
// a pair i < j of the window is defined iff vx vy > 0 over the samples called in both, and then
//   q = rint(2^32 r^2)   (r^2 as in LD pruning, uint64, round to nearest even; q <= 2^32).
// Every sum below is of q's and pair counts, so it is an exact integer: the kernels may add in any order, and the results
// are a function of the window's rows alone.  k_ld_windows leaves per row j, population p:
//   c_j = sum_{i < j} q (pairs whose larger row is j) and its count, written once by the CTA of j's block;
//   d_i = sum_{j > i} q (pairs whose smaller row is i) and its count, added with one atomic per (row, population, CTA);
//   the site bits.
// k_ldw_finish (one warp per window) turns them into n_sites, n_pairs, zns = 2^-32 sum q / n_pairs and, for each split
// after the k-th site s_k (row r_k), 2 <= k <= m - 2, with T = sum c over the window:
//   WL = sum_{j <= r_k} c_j,  P = sum_{i <= r_k} d_i,  WR = T - P,  X = P - WL   (and the same for the counts),
//   omega_k = ((WL + WR) / (nL + nR)) / (X / nX),  eligible iff nL + nR > 0 and X > 0; omega = the largest, lowest k on ties.
struct LdwParams {
  const uint32_t* G;           // B32 genotype matrix
  long long S;
  int W1, W2, ns1, ns2;
  const uint8_t* flags;        // snp_flags (NULL: every row passes, every row counted)
  const int32_t* pos;
  SegList seg;                 // candidate windows in row order (wlo, whi, ncand); segoff unused
  unsigned long long* c;       // [2][S] c_j of population 1, then 2
  unsigned long long* d;       // [2][S] d_i (zeroed before k_ld_windows)
  uint32_t* cn;                // [2][S] pairs counted in c_j
  uint32_t* dn;                // [2][S] pairs counted in d_i (zeroed)
  uint8_t* site;               // [S] bit p: row passes the filter and is a site of population p + 1
  int32_t* snp_count;          // [ncand] outputs
  uint8_t* out_flags;
  int32_t* n_sites[2];
  long long* n_pairs[2];
  double* zns[2];
  double* omega[2];
  long long* omega_pos[2];
};

__device__ __forceinline__ bool ldw_pass(const LdwParams& p, long long s) { return !p.flags || (__ldg(p.flags + s) & 1); }

// First row of the candidate window that holds row j, -1 when none does (the rows after a chromosome's last full
// fixed-SNP window).  Windows are disjoint and in row order; an empty window has wlo = whi, so the last window with
// wlo <= j is the only one that can hold j.
__device__ __forceinline__ long long ldw_window_start(const LdwParams& p, long long j) {
  if (p.seg.ncand == 0 || __ldg(p.seg.wlo) > j) return -1;
  long long lo = 0, hi = p.seg.ncand;
  while (hi - lo > 1) {
    const long long mid = (lo + hi) >> 1;
    if (__ldg(p.seg.wlo + mid) <= j) lo = mid; else hi = mid;
  }
  return j < __ldg(p.seg.whi + lo) ? __ldg(p.seg.wlo + lo) : -1;
}

struct LdSums {
  int n, ax, bx, ay, by, pp;
};

// The sums of k_ld_pairs (9 popcounts per word pair) of the LD_IROWS staged rows i from row0 with the staged row j = lane,
// over the staged word pairs [qa, qb).
__device__ __forceinline__ void ldw_sums(const uint32_t* sj, const uint4* si, int qa, int qb, int lane, int row0,
                                         LdSums (&s)[LD_IROWS]) {
#pragma unroll 4
  for (int q = qa; q < qb; ++q) {
    const uint32_t cy = sj[(q * 3 + 0) * BLK + lane], d1y = sj[(q * 3 + 1) * BLK + lane], d2y = sj[(q * 3 + 2) * BLK + lane];
#pragma unroll
    for (int k = 0; k < LD_IROWS; ++k) {
      const uint4 x = si[q * BLK + row0 + k];
      s[k].n += __popc(x.x & cy);
      s[k].ax += __popc(x.y & cy);
      s[k].bx += __popc(x.z & cy);
      s[k].ay += __popc(d1y & x.x);
      s[k].by += __popc(d2y & x.x);
      s[k].pp += __popc(x.y & d1y) + __popc(x.y & d2y) + __popc(x.z & d1y) + __popc(x.z & d2y);
    }
  }
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One CTA per 32-row block of rows j, staged as in k_ld_pairs; it streams the 32-row blocks of rows i from the one that
// holds the window start of its first row in a window up to its own block.  The word pairs of population 1 ([0, W1 / 2))
// and population 2 ([W1 / 2, NP)) go to separate sums.  The diagonal tile (i = j) gives each row's vx over its own calls:
// the site bits.
template <int TW1, int TW2>
__global__ void __launch_bounds__(LD_WARPS * 32) k_ld_windows(const __grid_constant__ LdwParams p) {
  constexpr int TNP = (TW1 + TW2) / 2;  // word pairs per row; 0: runtime
  __shared__ uint32_t sj[LD_KP * 3 * BLK];
  __shared__ uint4 si[LD_KP * BLK];
  __shared__ unsigned long long sc[LD_WARPS][2][BLK];
  __shared__ uint32_t scn[LD_WARPS][2][BLK];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int NP = TNP > 0 ? TNP : (p.W1 + p.W2) >> 1, RW = 2 * NP, H1 = TNP > 0 ? TW1 / 2 : p.W1 >> 1;
  const int nch = (NP + LD_KP - 1) / LD_KP;
  const long long jb = blockIdx.x, j0 = jb * BLK, j = j0 + lane;
  const bool jok = j < p.S;
  const long long wj = jok && ldw_pass(p, j) ? ldw_window_start(p, j) : -1;  // -1: row j is in no tested pair
  long long first = wj >= 0 ? wj : j0;
#pragma unroll
  for (int o = 16; o; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));

  auto stage_j = [&](int q0, int nq) {
    for (int t = threadIdx.x; t < nq * BLK; t += blockDim.x) {
      const int q = t >> 5, r = t & 31;
      const uint3 v = ld_planes(p, jb, RW, q0 + q, r);
      sj[(q * 3 + 0) * BLK + r] = v.x;
      sj[(q * 3 + 1) * BLK + r] = v.y;
      sj[(q * 3 + 2) * BLK + r] = v.z;
    }
  };
  if (nch == 1) stage_j(0, NP);

  unsigned long long csum[2] = {0ull, 0ull};
  uint32_t ccnt[2] = {0u, 0u};
  uint32_t site = 0u;
  for (long long ib = first >> 5; ib <= jb; ++ib) {
    const long long i0 = ib * BLK + warp * LD_IROWS;
    bool any = false;
#pragma unroll
    for (int k = 0; k < LD_IROWS; ++k) any |= (wj >= 0 && i0 + k >= wj && i0 + k < j) || (jok && i0 + k == j);
    any = __any_sync(0xffffffffu, any);
    LdSums s1[LD_IROWS], s2[LD_IROWS];
#pragma unroll
    for (int k = 0; k < LD_IROWS; ++k) s1[k] = s2[k] = LdSums{0, 0, 0, 0, 0, 0};
    for (int ch = 0; ch < nch; ++ch) {
      const int q0 = ch * LD_KP, nq = TNP > 0 ? TNP : min(LD_KP, NP - q0);
      __syncthreads();  // the previous pass's readers of sj / si are done
      if (nch > 1) stage_j(q0, nq);
      for (int t = threadIdx.x; t < nq * BLK; t += blockDim.x) {
        const int q = t >> 5, r = t & 31;
        const uint3 v = ld_planes(p, ib, RW, q0 + q, r);
        si[q * BLK + r] = make_uint4(v.x, v.y, v.z, 0u);
      }
      __syncthreads();
      if (!any) continue;
      const int qa = min(max(H1 - q0, 0), nq);  // staged pairs [0, qa) are population 1's
      ldw_sums(sj, si, 0, qa, lane, warp * LD_IROWS, s1);
      ldw_sums(sj, si, qa, nq, lane, warp * LD_IROWS, s2);
    }
    if (!any) continue;
#pragma unroll
    for (int k = 0; k < LD_IROWS; ++k) {
      const long long i = i0 + k;
      const bool tested = wj >= 0 && i >= wj && i < j && ldw_pass(p, i);
#pragma unroll
      for (int pop = 0; pop < 2; ++pop) {
        const LdSums& s = pop ? s2[k] : s1[k];
        const long long nn = s.n, sx = s.ax + s.bx, sy = s.ay + s.by;
        const long long cov = nn * s.pp - sx * sy;
        const unsigned long long vx = (unsigned long long)(nn * (s.ax + 3LL * s.bx) - sx * sx);
        const unsigned long long vy = (unsigned long long)(nn * (s.ay + 3LL * s.by) - sy * sy);
        const unsigned long long den = vx * vy;
        if (jok && i == j && vx > 0) site |= 1u << pop;  // i = j: vx over row j's own calls
        unsigned long long q = 0;
        const uint32_t one = tested && den > 0;
        if (one) {
          const unsigned long long ac = (unsigned long long)(cov < 0 ? -cov : cov);
          q = __double2ull_rn(__ull2double_rn(ac * ac) / __ull2double_rn(den) * 4294967296.0);  // exact scaling by 2^32
        }
        csum[pop] += q;
        ccnt[pop] += one;
        const uint32_t nd = __reduce_add_sync(0xffffffffu, one);
        if (nd) {  // warp-uniform
          const unsigned long long dq = warp_sum_u64(q);
          if (lane == 0) {
            atomicAdd(p.d + pop * p.S + i, dq);
            atomicAdd(p.dn + pop * p.S + i, nd);
          }
        }
      }
    }
  }
#pragma unroll
  for (int pop = 0; pop < 2; ++pop) {
    sc[warp][pop][lane] = csum[pop];
    scn[warp][pop][lane] = ccnt[pop];
  }
  if (jok && warp == lane / LD_IROWS) p.site[j] = (uint8_t)(ldw_pass(p, j) ? site : 0u);
  __syncthreads();
  if (warp < 2 && jok) {
    unsigned long long cs = 0;
    uint32_t cc = 0;
#pragma unroll
    for (int w = 0; w < LD_WARPS; ++w) {
      cs += sc[w][warp][lane];
      cc += scn[w][warp][lane];
    }
    p.c[warp * p.S + j] = cs;
    p.cn[warp * p.S + j] = cc;
  }
}

typedef unsigned __int128 u128;

// Round to nearest even: the bits below the top 64 fold into a sticky bit 0, far below the rounding position of the
// 64 -> 53-bit conversion, then an exact power-of-two scaling.
__device__ __forceinline__ double u128_to_double_rn(u128 v) {
  const unsigned long long hi = (unsigned long long)(v >> 64);
  if (hi == 0) return __ull2double_rn((unsigned long long)v);
  const unsigned long long lo = (unsigned long long)v;
  const int sh = 64 - __clzll((long long)hi);  // 1 .. 64: top = v >> sh has its bit 63 set
  const unsigned long long top = sh == 64 ? hi : (hi << (64 - sh)) | (lo >> sh);
  const bool sticky = sh == 64 ? lo != 0 : (lo << (64 - sh)) != 0;
  return __ull2double_rn(top | (sticky ? 1ull : 0ull)) * __longlong_as_double((long long)(1023 + sh) << 52);  // * 2^sh
}

__device__ __forceinline__ u128 shfl_u128(u128 v, int src, bool up, int delta) {
  const unsigned long long lo = (unsigned long long)v, hi = (unsigned long long)(v >> 64);
  const unsigned long long a = up ? __shfl_up_sync(0xffffffffu, lo, delta) : __shfl_sync(0xffffffffu, lo, src);
  const unsigned long long b = up ? __shfl_up_sync(0xffffffffu, hi, delta) : __shfl_sync(0xffffffffu, hi, src);
  return ((u128)b << 64) | a;
}

// Inclusive warp scans.
__device__ __forceinline__ u128 scan_u128(u128 v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u128 t = shfl_u128(v, 0, true, o);
    if (lane >= o) v += t;
  }
  return v;
}
__device__ __forceinline__ unsigned long long scan_u64(unsigned long long v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}

constexpr int LDW_FIN_WARPS = 8;  // warps per CTA of k_ldw_finish: one warp per window

// One warp per window: totals T, N and the sites first, then the splits in row order, 32 rows per step, with the prefix
// sums of c, d and their counts carried from step to step.  Lane-local best split (strict >, rows ascending: the lowest k),
// then a warp arg-max with the same tie rule.
__global__ void __launch_bounds__(LDW_FIN_WARPS * 32) k_ldw_finish(const __grid_constant__ LdwParams p) {
  const long long w = (long long)blockIdx.x * LDW_FIN_WARPS + (threadIdx.x >> 5);
  if (w >= p.seg.ncand) return;
  const int lane = threadIdx.x & 31;
  const long long lo = __ldg(p.seg.wlo + w), hi = __ldg(p.seg.whi + w);
  const double nan = __longlong_as_double(0x7FF8000000000000LL);
  int cnt = 0;
  for (long long r = lo + lane; r < hi; r += 32) cnt += p.flags ? (__ldg(p.flags + r) >> 1) & 1 : 1;
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  for (int pop = 0; pop < 2; ++pop) {
    const unsigned long long* C = p.c + pop * p.S;
    const unsigned long long* D = p.d + pop * p.S;
    const uint32_t* CN = p.cn + pop * p.S;
    const uint32_t* DN = p.dn + pop * p.S;
    u128 T = 0;
    unsigned long long N = 0;
    int m = 0;
    for (long long r = lo + lane; r < hi; r += 32) {
      T += C[r];
      N += CN[r];
      m += (p.site[r] >> pop) & 1;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      T += shfl_u128(T, lane ^ o, false, 0);
      N += __shfl_xor_sync(0xffffffffu, N, o);
    }
    m = __reduce_add_sync(0xffffffffu, m);
    double best = -1.0;  // every eligible omega is >= 0
    int best_k = 0;
    long long best_row = -1;
    if (m >= 4) {
      u128 wl0 = 0, p0 = 0;  // prefix sums over the rows before this step
      unsigned long long nl0 = 0, np0 = 0;
      int k0 = 0;
      for (long long base = lo; base < hi; base += 32) {
        const long long r = base + lane;
        const bool ok = r < hi;
        const bool is_site = ok && ((p.site[r] >> pop) & 1);
        const u128 WL = wl0 + scan_u128(ok ? C[r] : 0ull, lane);
        const u128 P = p0 + scan_u128(ok ? D[r] : 0ull, lane);
        const unsigned long long nL = nl0 + scan_u64(ok ? CN[r] : 0u, lane);
        const unsigned long long nP = np0 + scan_u64(ok ? DN[r] : 0u, lane);
        const unsigned sites = __ballot_sync(0xffffffffu, is_site);
        const int k = k0 + __popc(sites & (0xffffffffu >> (31 - lane)));
        if (is_site && k >= 2 && k <= m - 2) {
          const u128 WR = T - P, X = P - WL;
          const unsigned long long nR = N - nP, nX = nP - nL;
          if (nL + nR > 0 && X > 0) {
            const double om = (u128_to_double_rn(WL + WR) / __ull2double_rn(nL + nR)) /
                              (u128_to_double_rn(X) / __ull2double_rn(nX));
            if (om > best) { best = om; best_k = k; best_row = r; }
          }
        }
        wl0 = shfl_u128(WL, 31, false, 0);
        p0 = shfl_u128(P, 31, false, 0);
        nl0 = __shfl_sync(0xffffffffu, nL, 31);
        np0 = __shfl_sync(0xffffffffu, nP, 31);
        k0 += __popc(sites);
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int ok_ = __shfl_xor_sync(0xffffffffu, best_k, o);
        const long long orow = __shfl_xor_sync(0xffffffffu, best_row, o);
        if (ob > best || (ob == best && ok_ < best_k)) { best = ob; best_k = ok_; best_row = orow; }
      }
    }
    if (lane == 0) {
      p.n_sites[pop][w] = m;
      p.n_pairs[pop][w] = (long long)N;
      p.zns[pop][w] = N ? u128_to_double_rn(T) * 0x1p-32 / __ull2double_rn(N) : nan;
      p.omega[pop][w] = best_row >= 0 ? best : nan;
      p.omega_pos[pop][w] = best_row >= 0 ? (long long)__ldg(p.pos + best_row) : -1;
    }
  }
  if (lane == 0) {
    p.snp_count[w] = cnt;
    p.out_flags[w] = hi == lo ? TDSFS_F_EMPTY : 0;
  }
}

}  // namespace tdsfs
