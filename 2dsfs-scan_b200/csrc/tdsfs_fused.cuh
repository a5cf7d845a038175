// tdsfs_fused.cuh -- the fused scan of the genotype-level entry (DESIGN.md section 3):
//
//   k1_fused    ONE pass over the 2-bit genotype matrix does everything that does not need the final background:
//               per-SNP counts -> joint fold -> record store -> background histograms (as the plain count kernel), AND the
//               background-independent half of every window's statistics.  With
//                   T = 2 ( sum_bins x ln x  -  sum_SNPs ln b[bin_s]  -  N (ln N - ln B) )
//               (algebraically the reference's 2 (logpmf(x; x/N) - logpmf(x; b/B)), twoDSFS_class.py:625-684, :478-537)
//               the first sum and N depend on the window alone.  Every warp owns a CONTIGUOUS range of SNPs whose ends are
//               snapped to window starts, streams it through its own TMA stage (genotype tile + the tile's positions), finds
//               the window of each SNP from its position ((pos-1)//W, :898) or its rank in the chromosome (:1515-1535), and
//               keeps the current window's spectra in warp-private shared-memory tables: an open-addressing table of 2D bins
//               whose insert returns the bin's old count c (the sum grows by dx[c] = (c+1) ln(c+1) - c ln c) and packed
//               16-bit folded 1D bins walked when the window closes.  Per window it leaves {sum2D, sum1D_p1, sum1D_p2, N's}.
//   k3_finish   after the background is final (all-reduce + ln tables): per window, the gather sum_SNPs ln b[bin_s] over the
//               window's records and the three statistics.  The spectra for which the reference returns exactly 0.0 (a window
//               that is its own background, a window with one populated bin) are re-scored per bin.  Windows larger than the
//               warp tables (> WCAP SNPs) are scored by the CTA path over dense scratch in the same launch.
#pragma once
#include <type_traits>

#include "tdsfs_kernels.cuh"

namespace tdsfs {

// meta word of a window's sums: count_snps in bits 0..9, then the flags
constexpr uint32_t WS_ONE_2D = 1u << 10, WS_ONE_1A = 1u << 11, WS_ONE_1B = 1u << 12, WS_NALL = 1u << 13;

struct FusedParams {
  KeyParams k;
  int wmode;                  // 0 = no window sums (plain count kernel), 1 = fixed-bp windows, 2 = fixed-SNP windows
  uint32_t W, Wmagic;         // window size (bp or SNPs) and min(floor(2^32 / W), 2^32 - 1)
  const long long* cand_off;  // [C+1] first candidate window of every chromosome
  long long ncand;
  double* ws;                 // [ncand][4] = sum2D, sum1D_p1, sum1D_p2, bits(N2 | N1a << 10 | N1b << 20, meta)
  const double* dxI;          // dx[m] = (m+1) ln(m+1) - m ln m, m < LN_TABLE
  const double* lnI;          // ln m
  int pos_tma;                // the tile's positions ride the TMA ring (16-byte aligned position array)
  int tab_words;              // per-warp window tables: HASH_SLOTS + packed 1D words, a multiple of 4
  int nw1, nw2;               // packed 1D words per population: (n + 2) / 2
  // tail of the launch (single-launch passes with the peer exchange mapped): after a grid-wide barrier the resident CTAs
  // exchange the background with the other ranks through peer memory and build its ln tables: no separate launches
  int tail;
  unsigned int* gridbar;
  long long tail_timeout;
  FinParams fin;
  PeerParams peer;
  unsigned long long* epoch_mem;
  unsigned long long* stamps;     // diagnostics: clock64 of CTA 0 at the phases of the tail (null = off)
};

// dx[m] = (m+1) ln(m+1) - m ln m, written as ln(m+1) + m log1p(1/m) so that no large terms cancel
__global__ void k_dx_table(double* t, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) t[i] = i ? log((double)i + 1.0) + (double)i * log1p(1.0 / (double)i) : 0.0;
}

// exact x / W for x < 2^32 with M = min(floor(2^32 / W), 2^32 - 1): the estimate is at most one short
__device__ __forceinline__ uint32_t udiv_magic(uint32_t x, uint32_t W, uint32_t M) {
  uint32_t qd = __umulhi(x, M);
  if (x - qd * W >= W) ++qd;
  return qd;
}

struct ChromWin {
  int c = -1, lo = 0, hi = -1;  // chromosome and its row range
  int cbase = 0;                // first candidate window of the chromosome
  int nfull = 0;                // fixed-SNP mode: number of full windows
};

__device__ __forceinline__ void chrom_win(const FusedParams& q, int s, ChromWin& cw) {
  if (s >= cw.lo && s < cw.hi) return;
  const KeyParams& p = q.k;
  int lo = 0, hi = p.C;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(p.chrom_off + mid) <= s) lo = mid; else hi = mid;
  }
  cw.c = lo;
  cw.lo = (int)__ldg(p.chrom_off + lo);
  cw.hi = (int)__ldg(p.chrom_off + lo + 1);
  cw.cbase = (int)__ldg(q.cand_off + lo);
  cw.nfull = q.wmode == 2 ? (int)((uint32_t)(cw.hi - cw.lo) / q.W) : 0;
}

// candidate-window id of SNP s at position pv; -1 = in no window (tail of a chromosome in fixed-SNP mode)
__device__ __forceinline__ int window_id(const FusedParams& q, int s, int pv, ChromWin& cw) {
  chrom_win(q, s, cw);
  int id;
  if (q.wmode == 1) {
    id = cw.cbase + (int)udiv_magic(pv > 0 ? (uint32_t)(pv - 1) : 0u, q.W, q.Wmagic);  // pos 0 falls in window 0 (Q10)
  } else {
    const int j = (int)udiv_magic((uint32_t)(s - cw.lo), q.W, q.Wmagic);
    id = j < cw.nfull ? cw.cbase + j : -1;
  }
  return (long long)id < q.ncand ? id : -1;  // unsorted positions must not write out of bounds
}

// first row after `t` (within WCAP rows, same chromosome or its end) that starts another window than window k of row t;
// -1 when the window runs on beyond that (warp-cooperative, fixed-bp windows)
__device__ __forceinline__ int next_window_start(const FusedParams& q, int t, int k, ChromWin& cw, int lane) {
  const KeyParams& p = q.k;
  constexpr int STEP = WCAP / 32;  // 24
  auto past = [&](int s) -> bool { return s >= cw.hi || window_id(q, s, __ldg(p.pos + s), cw) != k; };
  const bool o1 = past(t + STEP * (lane + 1));
  const uint32_t b1 = __ballot_sync(0xffffffffu, o1);
  if (b1 == 0u) return -1;
  const int f = __ffs(b1) - 1;  // the start lies in (t + STEP f, t + STEP (f + 1)]
  const int base = t + STEP * f + 1;
  const bool o2 = lane < STEP ? past(base + lane) : true;
  const uint32_t b2 = __ballot_sync(0xffffffffu, o2);
  return min(base + __ffs(b2) - 1, cw.hi);
}

// Snap a range boundary `t` (a tile-aligned row) to the nearest window start, so that no window of at most WCAP SNPs is split
// between two warps (warp-cooperative: all lanes call, all return the same value; monotone in t).  Nearest rather than
// "back to the start of the window that holds t": the ranges of a small shard are only a few windows long, and their
// lengths then differ by at most one window instead of two.  nearest = false snaps back instead: the two ends of a launch,
// because rows past the end may still be uploading.
// is_start = the returned row starts a window (or lies in none); false when the window holding t began more than WCAP rows
// earlier and t itself is returned (such a window is larger than the warp tables: nobody sums it here, the CTA path scores
// it).  nearest returns t there only when the window also ends more than WCAP rows later; otherwise its end, which keeps
// the snapped boundaries monotone.
__device__ __forceinline__ int snap_row(const FusedParams& q, int t, bool& is_start, int lane, bool nearest) {
  const KeyParams& p = q.k;
  is_start = true;
  if (t <= 0) return 0;
  if (t >= (int)p.S) return (int)p.S;
  if (q.wmode == 0) return t;
  ChromWin cw;
  chrom_win(q, t, cw);
  if (t == cw.lo) return t;
  if (q.wmode == 2) {
    const int j = (int)udiv_magic((uint32_t)(t - cw.lo), q.W, q.Wmagic);
    if (j >= cw.nfull) return t;  // tail of the chromosome: no window
    if (q.W > (uint32_t)WCAP) {
      is_start = (t - cw.lo) == j * (int)q.W;
      return t;
    }
    const int back = cw.lo + j * (int)q.W, fwd = back + (int)q.W;  // fwd <= cw.hi: window j is a full one
    return (!nearest || (t - back) <= (fwd - t)) ? back : fwd;
  }
  const int k = window_id(q, t, __ldg(p.pos + t), cw);
  const int lo = max(cw.lo, t - WCAP);
  const int span = t - lo;               // 1 .. WCAP
  const int step = (span + 31) >> 5;     // 1 .. 24
  int back;
  // round 1: lanes probe lo + lane * step (window ids are monotone in the row: false ... false true ... true, t is true)
  const int s1 = lo + lane * step;
  const bool in1 = s1 < t ? window_id(q, s1, __ldg(p.pos + s1), cw) == k : true;
  const uint32_t b1 = __ballot_sync(0xffffffffu, in1);
  const int f = __ffs(b1) - 1;
  if (b1 == 0u) {                        // every probe lies before the window: it starts in (lo + 31 step, t]
    const int base = lo + 31 * step + 1;
    const int sc = base + lane;
    const bool in2 = sc < t ? window_id(q, sc, __ldg(p.pos + sc), cw) == k : true;
    const uint32_t b2 = __ballot_sync(0xffffffffu, in2);
    back = min(base + __ffs(b2) - 1, t);
  } else if (f == 0) {                   // row lo already belongs to the window
    if (lo != cw.lo) {                   // ... and it began even earlier: larger than WCAP rows
      // nearest: the window's end when it lies within WCAP rows.  An earlier target of this window may have snapped forward
      // to that end, and returning t < end would then hand rows [t, end) to two warps (counted twice in the background)
      if (nearest) {
        const int fwd = next_window_start(q, t, k, cw, lane);
        if (fwd >= 0) return fwd;
      }
      is_start = false;
      return t;
    }
    back = lo;                           // ... because the chromosome starts there
  } else {                               // round 2: the start lies in (lo + (f-1) step, lo + f step]
    const int base = lo + (f - 1) * step + 1;
    const int sc = base + lane;
    const int top = min(lo + f * step, t);
    const bool in2 = sc < top ? window_id(q, sc, __ldg(p.pos + sc), cw) == k : true;
    const uint32_t b2 = __ballot_sync(0xffffffffu, in2);
    back = min(base + __ffs(b2) - 1, top);
  }
  if (back == t || !nearest) return back;
  const int fwd = next_window_start(q, t, k, cw, lane);
  return (fwd < 0 || (t - back) <= (fwd - t)) ? back : fwd;
}

// ---- population counts of one SNP from its bit planes (compile-time word counts)
// sum of the popcounts of N words with carry-save adders: three words become a sum word (same weight) and a carry word (twice
// the weight), level by level, until at most two words per weight are left - one POPC each.  N = 7: 3 adders + 4 POPC,
// N = 16: 9 adders + 7 POPC (a POPC per word would be 16 of the slow pipe).
template <int N>
__device__ __forceinline__ uint32_t popc_sum(const uint32_t (&w)[N]) {
  if constexpr (N == 1) {
    return __popc(w[0]);
  } else if constexpr (N == 2) {
    return __popc(w[0]) + __popc(w[1]);
  } else {
    constexpr int M = N / 3, R = N - 3 * M;
    uint32_t ones[M + R], twos[M];
#pragma unroll
    for (int i = 0; i < M; ++i) csa(twos[i], ones[i], w[3 * i], w[3 * i + 1], w[3 * i + 2]);
#pragma unroll
    for (int i = 0; i < R; ++i) ones[M + i] = w[3 * M + i];
    return popc_sum<M + R>(ones) + 2u * popc_sum<M>(twos);
  }
}

// alt allele count and missing-call count of one population block (TW words = TW / 2 (lo, hi) pairs) of the lane's SNP:
// codes 00, 01, 11, 10 = hom-ref, het, hom-alt, missing  =>  alt = popc(lo) + popc(lo & hi), missing = popc(hi) - popc(lo & hi).
// Three bit-sliced counters over TW / 2 words each instead of one over all TW words plus one over the missing planes.
template <int TW>
__device__ __forceinline__ void count_pop_planes(const uint32_t* blk, uint32_t& alt, uint32_t& miss) {
  constexpr int P = TW / 2;
  uint32_t lo[P], hi[P], both[P];
#pragma unroll
  for (int i = 0; i < P; ++i) {
    lo[i] = blk[(2 * i) * BLK];
    hi[i] = blk[(2 * i + 1) * BLK];
    both[i] = lo[i] & hi[i];
  }
  const uint32_t c = popc_sum<P>(both);
  alt = popc_sum<P>(lo) + c;
  miss = popc_sum<P>(hi) - c;
}

// folded bin of a raw alt count, 0 when it does not enter the 1D likelihood (same values as folded_interior, fewer instructions)
__device__ __forceinline__ uint32_t fold_fast(int a, int n) {
  const uint32_t f = (uint32_t)min(a, 2 * n - a);
  return (f - 1u) < (uint32_t)(n - 1) ? f : 0u;
}

// predicated reductions without a branch (a divergent branch costs more than the reduction it skips)
__device__ __forceinline__ void red_shared_inc_if(bool pr, const uint32_t* base, uint32_t idx) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p red.shared.add.u32 [%1], 1;\n\t}" ::"r"((uint32_t)pr), "r"(smem_u32(base) + idx * 4u) : "memory");
}
__device__ __forceinline__ void red_global_inc_if(bool pr, uint32_t* addr) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p red.global.add.u32 [%1], 1;\n\t}" ::"r"((uint32_t)pr), "l"(addr) : "memory");
}

// PLAIN = the common configuration, with every per-SNP branch that cannot trigger compiled out: no snp_flags / fix-ups, one
// background group for all rows (or none), no position restriction of the background, fold on, 4-byte records, no more
// sample columns than the declared panel (so no count can leave the spectrum), 32 <= n <= 1023 (the privatised corner is
// exactly 64 x 64 and every 1D bin is privatised).  Everything else takes the generic instantiation.
// most warps an instantiation may be launched with: wide compile-time rows keep more words in registers and never fit more
// than 16 warps beside their tiles and tables anyway
template <int TW1, int TW2>
constexpr int k1f_max_warps() { return (TW1 + TW2) >= 48 ? 16 : K1_CWARPS; }

template <int TW1, int TW2, bool PLAIN>
__global__ void __launch_bounds__(k1f_max_warps<TW1, TW2>() * 32, 1) k1_fused(const __grid_constant__ FusedParams q) {
  const KeyParams& p = q.k;
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31;
  // the warp index through a shuffle: the compiler then knows that everything derived from it (stage and barrier addresses,
  // tile numbers, the TMA operands) is warp-uniform and keeps it in uniform registers instead of electing lanes around UBLKCP
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int W1 = TW1 > 0 ? TW1 : p.W1, W2 = TW2 > 0 ? TW2 : p.W2;
  const int RW = W1 + W2;
  const int tile_rows = p.tile_blocks * BLK;
  const int stage_stride = p.stage_bytes + tile_rows * 4;  // genotype tile, then the tile's positions
  const int depth = p.nstage / p.cwarps;                   // stages per warp
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)p.nstage * stage_stride);
  SinkSmem sm;
  sm.corner = reinterpret_cast<uint32_t*>(full + ((p.nstage + 1) & ~1));
  sm.h1a = sm.corner + p.cr * p.cc;
  sm.h1b = sm.h1a + p.h1a;
  const int nhist = p.cr * p.cc + p.h1a + p.h1b;
  uint32_t* tab = sm.corner + ((nhist + 3) & ~3) + (size_t)warp * q.tab_words;  // hash table | 1D pop1 | 1D pop2
  uint32_t* w1a = tab + HASH_SLOTS;
  uint32_t* w1b = w1a + q.nw1;

  if (tid == 0) {
    for (int i = 0; i < p.nstage; ++i) mbar_init(full + i, 1);
    fence_barrier_init();
    if (q.stamps && blockIdx.x == 0) q.stamps[0] = (unsigned long long)clock64();
  }
  for (int i = tid; i < nhist; i += blockDim.x) sm.corner[i] = 0;
  if (q.wmode && warp < p.cwarps) {
    for (int i = lane; i < HASH_SLOTS; i += 32) tab[i] = EMPTY_KEY;
    for (int i = lane; i < q.nw1 + q.nw2; i += 32) w1a[i] = 0;
  }
  __syncthreads();

  // part jj of the launch's rows [r0, r1) starts at a tile-aligned row near r0 + (r1 - r0) jj / nparts
  const int r0 = (int)p.r0, r1 = (int)p.r1, S = (int)p.S;
  const int nparts = gridDim.x * p.cwarps;
  auto target = [&](int jj) -> int {
    if (jj <= 0) return r0;
    if (jj >= nparts) return r1;
    const long long t = r0 + (long long)(r1 - r0) * jj / nparts;
    return max(r0, (int)(t / tile_rows * tile_rows));
  };
  ChromCache cc;
  const int cta_group = PLAIN ? p.uniform_group : tile_group(p, target(blockIdx.x * p.cwarps), cc);

  if (warp < p.cwarps) {
    const int j = blockIdx.x * p.cwarps + warp;
    // Interior boundaries snap to the nearest window start; the ends of the launch snap BACK (rows past r1 may still be
    // uploading, and the next launch starts from the same back-snapped row), and everything stays between them.
    bool st0 = true, st1 = true, stl = true, sth = true;
    const int lo_clamp = r0 > 0 ? snap_row(q, r0, stl, lane, false) : 0;
    const int hi_clamp = r1 < S ? snap_row(q, r1, sth, lane, false) : S;
    int slo = lo_clamp, shi = hi_clamp;
    if (j > 0) {
      slo = snap_row(q, target(j), st0, lane, true);
      if (slo <= lo_clamp) { slo = lo_clamp; st0 = stl; }
      if (slo >= hi_clamp) { slo = hi_clamp; st0 = sth; }
    } else {
      st0 = stl;
    }
    if (j + 1 < nparts) {
      shi = snap_row(q, target(j + 1), st1, lane, true);
      if (shi <= lo_clamp) shi = lo_clamp;
      if (shi >= hi_clamp) shi = hi_clamp;
    }
    slo = __shfl_sync(0xffffffffu, slo, 0);  // (uniform already; the shuffle tells the compiler)
    shi = __shfl_sync(0xffffffffu, shi, 0);
    st0 = __shfl_sync(0xffffffffu, (int)st0, 0) != 0;
    if (slo < shi) {
      uint8_t* stages = smem + (size_t)warp * depth * stage_stride;
      uint64_t* bars = full + warp * depth;
      const long long block_words = (long long)RW * BLK;
      const int b_end = (r1 + BLK - 1) / BLK;  // blocks this launch may read (later ones may still be uploading)
      const int S4 = S & ~3;                   // positions below S4 come through TMA in whole 16-byte groups
      const int t_begin = slo / tile_rows, t_end = (shi - 1) / tile_rows + 1;
      const int t_whole = min(b_end, S4 / BLK) / p.tile_blocks;  // tiles below this one are whole, positions included
      const uint32_t gbytes_whole = (uint32_t)(p.tile_blocks * block_words * 4);
      const uint32_t pbytes_whole = q.pos_tma ? (uint32_t)tile_rows * 4u : 0u;
      auto issue = [&](int t, int slot) {  // lane 0 only
        const int blk0 = t * p.tile_blocks;
        uint32_t gbytes = gbytes_whole, pbytes = pbytes_whole;
        if (t >= t_whole) {  // the last tile of the launch / of the matrix
          const int nb = min(p.tile_blocks, b_end - blk0);
          gbytes = (uint32_t)(nb * block_words * 4);
          pbytes = q.pos_tma ? (uint32_t)max(0, min(nb * BLK, S4 - blk0 * BLK)) * 4u : 0u;
        }
        uint8_t* stage = stages + (size_t)slot * stage_stride;
        mbar_arrive_expect_tx(bars + slot, gbytes + pbytes);
        bulk_g2s_stream(stage, p.G + (long long)blk0 * block_words, gbytes, bars + slot);
        if (pbytes) bulk_g2s(stage + p.stage_bytes, p.pos + (long long)blk0 * BLK, pbytes, bars + slot);
      };
      if (lane == 0)
        for (int d = 0; d < depth; ++d)
          if (t_begin + d < t_end) issue(t_begin + d, d);
      int slot = 0;
      uint32_t ph = 0;

      // ---- state of the window the warp is in
      int cur_id = -2;                 // -2 = none yet, -1 = rows outside every window
      bool overflow = false;           // the window is not summed here (more than WCAP SNPs, or entered mid-way)
      bool pending_skip = !st0;
      int wcount = 0;
      int win_end_pos = 0, win_end_row = 0;  // rows below win_end_row at positions below win_end_pos are in window cur_id
      double w2 = 0.0;
      uint32_t nn = 0;                 // N2 | N1a << 10 | N1b << 20 (this lane's share)
      uint32_t aux = 0;                // distinct 2D bins | SNPs with a 2D key << 10 | count_snps flags << 20
      ChromWin cw;
      const uint32_t last = (uint32_t)p.bins2d - 1;
      constexpr uint32_t F10 = (1u << KEY_SHIFT) - 1;

      auto close_window = [&]() {
        __syncwarp();
        if (cur_id >= 0) {
          if (!overflow) {
            double a1 = 0.0, b1 = 0.0;
            uint32_t dd = 0;  // distinct folded 1D bins: pop1 | pop2 << 10
            for (int i = lane; i < q.nw1; i += 32) {
              const uint32_t v = w1a[i];
              if (v) {
                w1a[i] = 0;
                const uint32_t x0 = v & 0xFFFF, x1 = v >> 16;
                a1 = fma(u32_to_double(x0), __ldg(q.lnI + x0), a1);  // ln 0 and ln 1 are stored as 0
                a1 = fma(u32_to_double(x1), __ldg(q.lnI + x1), a1);
                dd += (x0 != 0) + (x1 != 0);
              }
            }
            for (int i = lane; i < q.nw2; i += 32) {
              const uint32_t v = w1b[i];
              if (v) {
                w1b[i] = 0;
                const uint32_t x0 = v & 0xFFFF, x1 = v >> 16;
                b1 = fma(u32_to_double(x0), __ldg(q.lnI + x0), b1);
                b1 = fma(u32_to_double(x1), __ldg(q.lnI + x1), b1);
                dd += ((x0 != 0) + (x1 != 0)) << 10;
              }
            }
            const uint32_t nt = __reduce_add_sync(0xffffffffu, nn);
            const uint32_t at = __reduce_add_sync(0xffffffffu, aux);
            const uint32_t dt = __reduce_add_sync(0xffffffffu, dd);
            const double w2t = warp_sum(w2);
            a1 = warp_sum(a1);
            b1 = warp_sum(b1);
            const uint32_t cft = PLAIN ? (uint32_t)wcount : (at >> 20);
            const uint32_t meta = cft | ((at & F10) == 1u ? WS_ONE_2D : 0u) | ((dt & F10) == 1u ? WS_ONE_1A : 0u) |
                                  ((dt >> 10) == 1u ? WS_ONE_1B : 0u) | (((at >> 10) & F10) ? WS_NALL : 0u);
            if (lane < 4) {
              const double v = lane == 0 ? w2t : (lane == 1 ? a1 : (lane == 2 ? b1 : __hiloint2double((int)meta, (int)nt)));
              q.ws[(long long)cur_id * 4 + lane] = v;
            }
          } else {
            for (int i = lane; i < q.nw1 + q.nw2; i += 32) w1a[i] = 0;
          }
          uint4* t4 = reinterpret_cast<uint4*>(tab);
#pragma unroll
          for (int i = 0; i < HASH_SLOTS / 128; ++i) t4[lane + i * 32] = make_uint4(EMPTY_KEY, EMPTY_KEY, EMPTY_KEY, EMPTY_KEY);
        }
        w2 = 0.0;
        nn = aux = 0;
        wcount = 0;
        __syncwarp();
      };

      // this lane's SNP enters the current window's tables (2D: the insert returns the bin's old count c)
      auto insert = [&](uint32_t key, uint32_t fa, uint32_t fb, uint32_t cf) {
        if (key != 0 && key != last) {
          uint32_t h = (key * 0x9E3779B1u) >> 22;  // HASH_SLOTS = 2^10
          const uint32_t fresh = (key << KEY_SHIFT) | 1u;
          uint32_t c;
          while (true) {  // most bins of a window are new: try to claim the slot first
            const uint32_t e = atomicCAS(tab + h, EMPTY_KEY, fresh);
            if (e == EMPTY_KEY) { c = 0; break; }
            if ((e >> KEY_SHIFT) == key) { c = atomicAdd(tab + h, 1u) & F10; break; }
            h = (h + 1) & (HASH_SLOTS - 1);
          }
          w2 += __ldg(q.dxI + c);  // dx[0] = 0: no branch for the (common) first SNP of a bin
          nn += 1u;
          aux += c == 0;
        }
        bump_half_if(w1a, fa);
        bump_half_if(w1b, fb);
        nn += (fa ? 1u << 10 : 0u) + (fb ? 1u << 20 : 0u);
        aux += (key != 0 ? 1u << 10 : 0u) + (PLAIN ? 0u : cf << 20);
      };

      int pv_next = 0;  // position of this lane's row in the next block (the path without the positions in the TMA ring)
      if (q.wmode == 1 && !q.pos_tma) {
        const int s_first = t_begin * tile_rows + lane;
        pv_next = s_first < S ? __ldg(p.pos + s_first) : 0;
      }
      // one 32-SNP block of the tile in the current stage.  INTERIOR (compile time) = the whole tile lies inside this warp's
      // range, which is every tile but the first and the last: no per-block range tests, positions always from the stage
      auto do_block = [&](auto interior_tag, int t, int blk0, int nb, int b, const uint32_t* tile, const int* spos) {
          constexpr bool INTERIOR = decltype(interior_tag)::value;
          const int sb = (blk0 + b) * BLK;
          const int s = sb + lane;
          const bool live = INTERIOR || (sb + BLK > slo && sb < shi);  // warp-uniform: the block holds rows of this warp's range
          uint32_t T1 = 0, M1 = 0, T2 = 0, M2 = 0;
          int pv = 0;
          if (live) {
            const uint32_t* rowp = tile + (size_t)b * block_words + lane;
            if constexpr (TW1 > 0 && TW2 > 0) {  // T = alt + missing, as the generic counter returns it
              count_pop_planes<TW1>(rowp, T1, M1);
              count_pop_planes<TW2>(rowp + TW1 * BLK, T2, M2);
              T1 += M1;
              T2 += M2;
            } else {
              count_block_b32<TW1>(rowp, W1, T1, M1);
              count_block_b32<TW2>(rowp + W1 * BLK, W2, T2, M2);
            }
            if (q.wmode == 1 && q.pos_tma) {
              if (INTERIOR || s < S4) pv = spos[b * BLK + lane];
              else if (s < S) pv = __ldg(p.pos + s);
            }
          }
          if (q.wmode == 1 && !q.pos_tma) {  // positions by plain loads, requested one block ahead (blocks come in row order)
            pv = pv_next;
            pv_next = s + BLK < S ? __ldg(p.pos + s + BLK) : 0;
          }
          if (b == nb - 1) {
            // the stage has been read completely: refill it BEFORE the fold / record / histogram / window work of its
            // last block, so that work overlaps the next load instead of delaying it
            __syncwarp();
            if (lane == 0 && t + depth < t_end) {
              fence_proxy_async();  // order this warp's generic-proxy reads of the stage before the async-proxy refill
              issue(t + depth, slot);
            }
          }
          if (!live) return;
          const bool whole = INTERIOR || (sb >= slo && sb + BLK <= shi);  // every lane's row belongs to this warp
          const bool act = whole || (s >= slo && s < shi);
          uint32_t key = 0, fa = 0, fb = 0, cf = 1;
          if (act) {
            const int alt1 = (int)(T1 - M1), alt2 = (int)(T2 - M2);
            const int ref1 = 2 * (p.ns1 - (int)M1) - alt1, ref2 = 2 * (p.ns2 - (int)M2) - alt2;
            if (PLAIN) {
              const bool swapped = alt1 + alt2 > p.n1 + p.n2;  // joint fold, twoDSFS_class.py:199-206
              const int k1 = swapped ? ref1 : alt1, k2 = swapped ? ref2 : alt2;
              int d1 = swapped ? (p.n1 - p.ns1) + (int)M1 : 0, d2 = swapped ? (p.n2 - p.ns2) + (int)M2 : 0;
              if ((d1 | d2) >> p.fmt.md) {  // does not fit the narrow record: the host redoes the pass with wide records
                atomicOr(p.err, 8);
                d1 = d2 = 0;
              }
              key = (uint32_t)(k1 * p.C2 + k2);  // (0,0) -> 0 : skipped SNP (:212)
              __stcs(reinterpret_cast<uint32_t*>(p.rec) + s,
                     (uint32_t)k1 | ((uint32_t)k2 << p.fmt.b1) | ((uint32_t)d1 << (p.fmt.b1 + p.fmt.b2)) |
                         ((uint32_t)d2 << (p.fmt.b1 + p.fmt.b2 + p.fmt.md)));
              fa = fold_fast(alt1, p.n1);
              fb = fold_fast(alt2, p.n2);
              if (cta_group >= 0) {  // background: privatised 64 x 64 corner and 1D bins, the rest straight to global memory
                const bool inc = (k1 | k2) < CORNER;
                red_shared_inc_if(key != 0 && inc, sm.corner, (uint32_t)(k1 << 6 | k2) & (CORNER * CORNER - 1));
                red_global_inc_if(key != 0 && !inc, p.hist + key);
                red_shared_inc_if(alt1 != 0, sm.h1a, (uint32_t)alt1);
                red_shared_inc_if(alt2 != 0, sm.h1b, (uint32_t)alt2);
              }
            } else {
              const uint2 ka = sink_row(p, s, ref1, alt1, ref2, alt2, cta_group, sm, cc);
              key = ka.x;
              fa = ka.y & 0xFFFF;
              fb = ka.y >> 16;
              if (p.flags) cf = (__ldg(p.flags + s) >> 1) & 1u;
            }
          }
          if (!q.wmode) return;
          // ---- window stage.  Fast path: every row of the block lies in the window the warp is already in
          if (whole && cur_id >= 0 && __all_sync(0xffffffffu, pv < win_end_pos && s < win_end_row)) {
            if (!overflow) {
              wcount += BLK;
              if (wcount > WCAP) overflow = true;
              else insert(key, fa, fb, cf);
            }
            return;
          }
          int wid = -1;
          if (act) wid = window_id(q, s, pv, cw);
          uint32_t rem = __ballot_sync(0xffffffffu, act);
          while (rem) {
            const int first = __ffs(rem) - 1;
            const int idf = __shfl_sync(0xffffffffu, wid, first);
            if (idf != cur_id) {
              close_window();
              cur_id = idf;
              overflow = pending_skip;
              pending_skip = false;
            }
            const bool mine = act && wid == idf;
            const uint32_t m = __ballot_sync(0xffffffffu, mine);
            rem &= ~m;
            if (cur_id >= 0 && !overflow) {
              wcount += __popc(m);
              if (wcount > WCAP) overflow = true;
              else if (mine) insert(key, fa, fb, cf);
            }
          }
          // extent of the window the warp is in now (that of the block's last active row)
          {
            const uint32_t am = __ballot_sync(0xffffffffu, act);
            const int src = 31 - __clz((int)am);  // am != 0: the block is live
            const int c_lo = __shfl_sync(0xffffffffu, cw.lo, src), c_hi = __shfl_sync(0xffffffffu, cw.hi, src);
            const int c_base = __shfl_sync(0xffffffffu, cw.cbase, src);
            if (cur_id < 0) {
              win_end_pos = 0;  // outside every window: keep taking the general path
              win_end_row = 0;
            } else if (q.wmode == 1) {
              const long long e = 1 + (long long)(cur_id - c_base + 1) * (long long)q.W;
              win_end_pos = e > 0x7FFFFFFFLL ? 0x7FFFFFFF : (int)e;
              win_end_row = c_hi;
            } else {
              win_end_pos = 0x7FFFFFFF;
              win_end_row = c_lo + (cur_id - c_base + 1) * (int)q.W;
            }
          }
      };

      for (int t = t_begin; t < t_end; ++t) {
        const int blk0 = t * p.tile_blocks;
        const int nb = min(p.tile_blocks, b_end - blk0);
        mbar_wait(bars + slot, ph);
        const uint8_t* stage = stages + (size_t)slot * stage_stride;
        const uint32_t* tile = reinterpret_cast<const uint32_t*>(stage);
        const int* spos = reinterpret_cast<const int*>(stage + p.stage_bytes);
        if (blk0 * BLK >= slo && (blk0 + nb) * BLK <= shi) {
          for (int b = 0; b < nb; ++b) do_block(std::true_type{}, t, blk0, nb, b, tile, spos);
        } else {
          for (int b = 0; b < nb; ++b) do_block(std::false_type{}, t, blk0, nb, b, tile, spos);
        }
        if (++slot == depth) { slot = 0; ph ^= 1; }
      }
      if (q.wmode) close_window();
    }
  }
  __syncthreads();
  sink_flush(p, sm, cta_group, tid, blockDim.x);
  if (q.tail) {
    // diagnostics (TDSFS_TAIL_STAMPS=1): clock64 of CTA 0 at [1] its histograms flushed, [2] past the grid barrier, [3..5] in
    // peer_exchange, [6] ln tables done, [7] totals done ([0] = kernel entry)
    auto stamp = [&](int i) { if (q.stamps && blockIdx.x == 0 && tid == 0) q.stamps[i] = (unsigned long long)clock64(); };
    stamp(1);
    grid_barrier(q.gridbar, p.err, q.tail_timeout);  // every CTA's private histograms are in the global histogram
    stamp(2);
    peer_exchange(q.peer, q.epoch_mem, q.stamps);
    for (int g = 0; g < q.fin.NG; ++g) finalize_tables(q.fin, g, blockIdx.x, gridDim.x);
    stamp(6);
    finalize_totals(q.fin, gridDim.x);
    stamp(7);
  }
}

// ------------------------------------------------------------------------------------------------ finish pass
struct FinishParams {
  ScoreParams s;
  const double* ws;   // window sums of k1_fused
  int use_smem;       // narrow records + one background group + a spectrum of at least 64 x 64: ln b tables in shared memory
  int large_ctas;     // CTAs (scratch slabs) of the large-window path
};

// bin of record r in spectrum `which` (0 = 2D, 1 = 1D pop1, 2 = 1D pop2); 0 = the SNP is not in that likelihood
__device__ __forceinline__ uint32_t bin_of(const uint2 r, int which, uint32_t last) {
  if (which == 0) return (r.x != 0 && r.x != last) ? r.x : 0u;
  return which == 1 ? (r.y & 0xFFFF) : (r.y >> 16);
}

// sum over the distinct bins of one spectrum of a window (cnt <= WCAP) of x (ln x - ln b), bin by bin as the reference's
// logpmf difference weighs them: O(cnt^2 / 32) per warp, used only for the windows that must reproduce an exact 0.0
__device__ __forceinline__ double exact_bins(const ScoreParams& p, int lo, int cnt, int which, const double* lb, int lane) {
  const uint32_t last = (uint32_t)p.bins2d - 1;
  double acc = 0.0;
  for (int ci = 0; ci < cnt; ci += 32) {
    const int i = ci + lane;
    const uint32_t ki = i < cnt ? bin_of(load_rec(p.rec, p.fmt, lo + i, p.n1, p.n2, p.C2), which, last) : 0u;
    uint32_t x = 0;
    bool earlier = false;
    for (int cj = 0; cj < cnt; cj += 32) {
      const int jn = cj + lane;
      const uint32_t kj = jn < cnt ? bin_of(load_rec(p.rec, p.fmt, lo + jn, p.n1, p.n2, p.C2), which, last) : 0u;
      for (int t = 0; t < 32; ++t) {
        const uint32_t kk = __shfl_sync(0xffffffffu, kj, t);
        const bool eq = kk == ki;
        x += eq;
        earlier |= eq && (cj + t < i);
      }
    }
    if (ki && !earlier) acc = fma(u32_to_double(x), (x > 1 ? ln_mult(p, x) : 0.0) - __ldg(lb + ki), acc);
  }
  return warp_sum(acc);
}

// Statistics of one small window from its background-dependent sums (g2, g1a, g1b: valid on every lane) and the window sums
// the count kernel left (wsv: lane l holds word l & 3 of the window's four).  Lanes 0..2 finish one statistic each.
__device__ __forceinline__ void finish_window(const ScoreParams& p, long long id, int lo, int cnt, double g2, double g1a, double g1b,
                                              double wsv, const double* lb2, const double* lb1a, const double* lb1b, const double* Bg,
                                              int lane) {
  const double bits = __shfl_sync(0xffffffffu, wsv, 3);
  const uint32_t nt = (uint32_t)__double2loint(bits), meta = (uint32_t)__double2hiint(bits);
  const int Nq = lane == 0 ? (int)(nt & 0x3FF) : (lane == 1 ? (int)((nt >> 10) & 0x3FF) : (int)(nt >> 20));
  const double Gq = lane == 0 ? g2 : (lane == 1 ? g1a : g1b);
  const bool one = lane < 3 && (meta & (WS_ONE_2D << lane)) != 0;
  const bool own = lane < 3 && Nq > 0 && (double)Nq == __ldg(Bg + lane);  // N == B: possibly the background itself
  double acc = wsv - Gq;
  const uint32_t exact = __ballot_sync(0xffffffffu, one || own) & 7u;
  if (exact) {  // per-bin form for the spectra where the reference's difference of logpmfs is exactly 0.0
    for (int w = 0; w < 3; ++w)
      if (exact & (1u << w)) {
        const double a = exact_bins(p, lo, cnt, w, w == 0 ? lb2 : (w == 1 ? lb1a : lb1b), lane);
        if (lane == w) acc = a;
      }
  }
  bool none = false;
  double Tq = 0.0;
  if (lane < 3) Tq = clr_value(p, Nq, acc, Bg, lane, none);
  const uint32_t nb = __ballot_sync(0xffffffffu, none) & 7u;  // bit q = statistic q is None
  if (lane == 0) {
    uint8_t f = (uint8_t)nb;  // TDSFS_F_T2D_NONE = 1, _P1_NONE = 2, _P2_NONE = 4
    if (p.snp_mode && !(meta & WS_NALL)) f |= TDSFS_F_SKIPPED;  // :1496 window skipped when its 2D spectrum sums to 0
    p.r_count[id] = (int)(meta & 0x3FF);
    p.r_flags[id] = f;
    p.r_T2[id] = Tq;
    p.r_n2[id] = Nq;
  } else if (lane == 1) {
    p.r_T1a[id] = Tq;
    p.r_n1a[id] = Nq;
  } else if (lane == 2) {
    p.r_T1b[id] = Tq;
    p.r_n1b[id] = Nq;
  }
}

__global__ void __launch_bounds__(256, 3) k3_finish(const __grid_constant__ FinishParams q) {
  // ln b of group 0 staged per CTA: [64 x 64] the low-count corner of the 2D table, entry 0 (the skipped bin) = 0, then the 1D
  // tables indexed by the UNFOLDED count a = k + 2 d of the narrow record (ln b[fold(a)], 0 where the SNP is not in the 1D
  // likelihood): the per-SNP work is two shifts, three table reads and three adds, without a fold or a validity branch
  extern __shared__ __align__(16) double sd[];
  const ScoreParams& p = q.s;
  const int lane = threadIdx.x & 31;
  const bool fast = q.use_smem != 0;  // host: narrow records, one background group, spectrum at least 64 x 64
  const uint32_t last = (uint32_t)p.bins2d - 1;
  const long long nwarp = (long long)gridDim.x * (blockDim.x >> 5);
  const long long wid = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (fast) {
    double* s_c = sd;
    double* s_a = sd + CORNER * CORNER;
    double* s_b = s_a + 2 * p.n1 + 1;
    for (int i = threadIdx.x; i < CORNER * CORNER; i += blockDim.x) s_c[i] = i ? __ldg(p.lb2 + (long long)(i >> 6) * p.C2 + (i & 63)) : 0.0;
    for (int i = threadIdx.x; i <= 2 * p.n1; i += blockDim.x) { const uint32_t f = fold_fast(i, p.n1); s_a[i] = f ? __ldg(p.lb1a + f) : 0.0; }
    for (int i = threadIdx.x; i <= 2 * p.n2; i += blockDim.x) { const uint32_t f = fold_fast(i, p.n2); s_b[i] = f ? __ldg(p.lb1b + f) : 0.0; }
    __syncthreads();
    const uint32_t m1 = (1u << p.fmt.b1) - 1u, m2 = (1u << p.fmt.b2) - 1u, md = (1u << p.fmt.md) - 1u;
    const int sh2 = p.fmt.b1, shd1 = p.fmt.b1 + p.fmt.b2, shd2 = p.fmt.b1 + p.fmt.b2 + p.fmt.md;
    const uint32_t* rec = reinterpret_cast<const uint32_t*>(p.rec);
    // ln b of one decoded record: the 2D read (shared-memory corner, else a gather from the L2-resident table) ...
    auto lookup2 = [&](uint32_t rr) -> double {
      const uint32_t k1 = rr & m1, k2 = (rr >> sh2) & m2;
      if ((k1 | k2) < (uint32_t)CORNER) return s_c[(k1 << 6) | k2];
      const uint32_t key = k1 * (uint32_t)p.C2 + k2;
      return key != last ? __ldg(p.lb2 + key) : 0.0;
    };
    // ... and the two 1D reads (shared memory)
    auto lookup1 = [&](uint32_t rr, double& la, double& lb) {
      const uint32_t k1 = rr & m1, k2 = (rr >> sh2) & m2;
      la = s_a[k1 + 2u * ((rr >> shd1) & md)];
      lb = s_b[k2 + 2u * (rr >> shd2)];
    };
    {
      // Windows dealt out round-robin; software pipeline over windows: while window i is processed, the first 256 records of
      // window i + 1 and the bounds of window i + 2 are in flight; a window's records beyond the first 256 are requested at
      // its start (one more batch) or on demand (above 512).
      constexpr int Q = 8;  // records per lane and batch
      auto bounds = [&](long long w, int& lo, int& cnt) {
        lo = 0; cnt = 0;
        if (w < p.ncand) {
          lo = __ldg(p.wlo + w);
          const int c = __ldg(p.whi + w) - lo;
          cnt = c <= WCAP ? c : 0;  // large windows are scored by the CTA path below
        }
      };
      auto load_batch = [&](uint32_t (&r)[Q], int lo, int cnt, int base) {
#pragma unroll
        for (int j = 0; j < Q; ++j) {
          const int i = base + j * 32 + lane;
          r[j] = i < cnt ? __ldcs(rec + lo + i) : 0u;  // 0 decodes to the skipped bin: every table holds 0 there
        }
      };
      double g2 = 0.0, g1a = 0.0, g1b = 0.0;
      auto consume = [&](const uint32_t (&r)[Q]) {
        // four records at a time: their reads are issued together, then accumulated (eight at a time measured 5 % slower)
#pragma unroll
        for (int h4 = 0; h4 < Q; h4 += 4) {
          double l2[4], la[4], lb[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            l2[j] = lookup2(r[h4 + j]);
            lookup1(r[h4 + j], la[j], lb[j]);
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) { g2 += l2[j]; g1a += la[j]; g1b += lb[j]; }
        }
      };
      long long id = wid, nid = wid + nwarp;
      int lo, cnt, nlo, ncnt;
      bounds(id, lo, cnt);
      bounds(nid, nlo, ncnt);
      uint32_t rn[Q];
      load_batch(rn, lo, cnt, 0);
      while (id < p.ncand) {
        uint32_t r[Q], r2[Q];
#pragma unroll
        for (int j = 0; j < Q; ++j) r[j] = rn[j];
        if (cnt > Q * 32) load_batch(r2, lo, cnt, Q * 32);
        const long long nnid = nid + nwarp;
        int nnlo, nncnt;
        bounds(nnid, nnlo, nncnt);
        load_batch(rn, nlo, ncnt, 0);
        if (cnt > 0) {
          const double wsv = __ldg(q.ws + id * 4 + (lane & 3));
          g2 = g1a = g1b = 0.0;
          consume(r);
          if (cnt > Q * 32) consume(r2);
          if (cnt > 2 * Q * 32) {
            load_batch(r2, lo, cnt, 2 * Q * 32);
            consume(r2);
          }
          g2 = warp_sum(g2); g1a = warp_sum(g1a); g1b = warp_sum(g1b);
          finish_window(p, id, lo, cnt, g2, g1a, g1b, wsv, p.lb2, p.lb1a, p.lb1b, p.B, lane);
        }
        id = nid; lo = nlo; cnt = ncnt;
        nid = nnid; nlo = nnlo; ncnt = nncnt;
      }
    }
  } else {
    for (long long id = wid; id < p.ncand; id += nwarp) {
      const int lo = __ldg(p.wlo + id), hi = __ldg(p.whi + id);
      const int cnt = hi - lo;
      if (cnt == 0 || cnt > WCAP) continue;  // empty: flagged by K2; large: the CTA path below
      const int g = p.score_group ? __ldg(p.score_group + __ldg(p.wchrom + id)) : 0;
      const double* lb2 = p.lb2 + (long long)g * p.bins2d;
      const double* lb1a = p.lb1a + (long long)g * (p.n1 + 1);
      const double* lb1b = p.lb1b + (long long)g * (p.n2 + 1);
      double g2 = 0.0, g1a = 0.0, g1b = 0.0;
      constexpr int Q = 4;
      for (int base = 0; base < cnt; base += Q * 32) {
        uint2 r[Q];
        double l2[Q], la[Q], lb[Q];
#pragma unroll
        for (int j = 0; j < Q; ++j) {
          const int i = base + j * 32 + lane;
          r[j] = i < cnt ? load_rec(p.rec, p.fmt, lo + i, p.n1, p.n2, p.C2) : make_uint2(0u, 0u);
        }
#pragma unroll
        for (int j = 0; j < Q; ++j) {
          const uint32_t key = r[j].x, fa = r[j].y & 0xFFFF, fb = r[j].y >> 16;
          l2[j] = (key != 0 && key != last) ? __ldg(lb2 + key) : 0.0;
          la[j] = fa ? __ldg(lb1a + fa) : 0.0;
          lb[j] = fb ? __ldg(lb1b + fb) : 0.0;
        }
#pragma unroll
        for (int j = 0; j < Q; ++j) { g2 += l2[j]; g1a += la[j]; g1b += lb[j]; }
      }
      g2 = warp_sum(g2); g1a = warp_sum(g1a); g1b = warp_sum(g1b);
      const double wsv = __ldg(q.ws + id * 4 + (lane & 3));
      finish_window(p, id, lo, cnt, g2, g1a, g1b, wsv, lb2, lb1a, lb1b, p.B + g * 6, lane);
    }
  }
  // windows above WCAP SNPs (K2's list, complete before this launch): one CTA each over dense scratch
  if ((int)blockIdx.x < q.large_ctas && *p.nlarge > 0) score_large_windows(p, blockIdx.x, min((int)gridDim.x, q.large_ctas));
}

}  // namespace tdsfs
