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

// Sample bits of word pair q (population 1's pairs, then population 2's) that are not padding.
__device__ __forceinline__ uint32_t ld_valid(const LdParams& p, int q) {
  const int h1 = p.W1 >> 1;
  const int left = q < h1 ? p.ns1 - 32 * q : p.ns2 - 32 * (q - h1);
  return left >= 32 ? 0xffffffffu : (left <= 0 ? 0u : (1u << left) - 1u);
}

// Planes of one 32-row B32 block's word pair q: called c = (lo | ~hi), d1 = lo (g >= 1), d2 = lo & hi (g = 2).  d1 and d2
// are 0 on missing calls; all three are masked to the pair's samples.
__device__ __forceinline__ uint3 ld_planes(const LdParams& p, long long blk, int RW, int q, int r) {
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

}  // namespace tdsfs
