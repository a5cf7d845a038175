// tdsfs_kernels.cuh -- hand-written sm_100a kernels of the 2DSFS-scan hot path.
//
// Reference code replaced (paths relative to uricchio/2DSFS-scan):
//   K1  count kernel        scripts/src/twoDSFS_class.py:118-130 (per-sample ref/alt counting),
//                           :190-217 (joint fold, skip, 2D bin), :427-433 (raw 1D alt count)
//   K2  window boundaries   :843-949 (fixed-bp walk), :1515-1535 (fixed-SNP walk)
//   K3  window spectra      :140-232, :398-463 applied to window_data
//   K4  fused scores        :478-537, :625-684 (scipy multinomial.logpmf difference)
//
// All integer work is exact; likelihoods are fp64.  No tensor cores (nothing here is a contraction).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/tdsfs.h"

namespace tdsfs {

// ------------------------------------------------------------------------------------------------ constants
constexpr int BLK = 32;               // SNPs per block of the block-transposed genotype layout ("B32", DESIGN.md)
constexpr int K1_CWARPS = 24;         // most warps the genotype count kernel can run (each runs its own TMA ring)
constexpr int K1_THREADS = K1_CWARPS * 32;  // launch bound; the launch uses cwarps * 32 threads
constexpr int K1_DEFAULT_WARPS = 12;
constexpr int K1_ROWS = 128;          // row granularity of host-side upload chunks (multiple of BLK)
constexpr int CORNER = 64;            // privatised low-count corner of the 2D background histogram (per CTA, smem)
constexpr int H1CAP = 2048;           // privatised 1D bins per population (per CTA, smem)
constexpr int HASH_SLOTS = 1024;      // per-warp open-addressing table of the window scorer
constexpr int WCAP = 768;             // windows up to WCAP SNPs are scored by one warp; larger ones by a CTA
constexpr int LN_TABLE = 4096;        // ln(m) lookup for window multiplicities
constexpr uint32_t EMPTY_KEY = 0xFFFFFFFFu;

// Per-SNP record written by the count kernels and read by the scorers.
//   wide   (uint2):   x = folded 2D bin a1' * (2n2+1) + a2' (0 = contributes nothing),
//                     y = fa | fb << 16: folded interior 1D bins of pop1 / pop2 (0 = not in that 1D likelihood)
//   narrow (uint32):  k1 | k2 << b1 | d1 << (b1+b2) | d2 << (b1+b2+md) with (k1, k2) = (a1', a2') the folded 2D cell and
//                     d = 0 for an unswapped SNP, (2n - alt - ref) / 2 (missing diploids) for a swapped one, so that the
//                     folded 1D bin is fold(k + 2d) either way (fold(a) = fold(2n - a)).  Half the bytes of the wide form;
//                     a SNP whose d does not fit `md` bits raises err bit 3 and the pass is redone with wide records.
struct RecFmt {
  int narrow, b1, b2, md;
};

struct KeyParams {
  int n1, n2, fold, C2, bins2d, R1, R2;   // R1 = 2n1+1, R2 = C2 = 2n2+1
  int ns1, ns2, W1, W2;                   // sample columns and uint32 words per population block
  long long S, r0, r1;                    // total rows; row range of this launch
  const uint32_t* G;
  const uint16_t* cnt;
  const int32_t* pos;
  const uint8_t* flags;
  const tdsfs_fixup_t* fix;
  long long nfix;
  void* rec;          // per-SNP records (RecFmt)
  RecFmt fmt;
  uint32_t* hist;     // [group][bins2d | R1 | R2]
  long long gstride;
  const int32_t* bg_group;  // per chromosome -> background group, -1 = not in any background; NULL = uniform_group
  int uniform_group;        // used when bg_group == NULL (0 = genome-wide, -1 = no background)
  const long long* chrom_off;
  int C;
  long long bg_lo, bg_hi;   // optional position restriction of the background (-1 = none)
  int* err;                 // bit0: count out of range, bit2: peer timeout, bit3: narrow record overflow
  int cr, cc;               // corner dims actually used: min(R1, CORNER), min(R2, CORNER)
  int h1a, h1b;             // privatised 1D bins: min(R1, H1CAP), min(R2, H1CAP)
  int nstage, stage_bytes;  // K1 ring: stages of `tile_blocks` 32-SNP blocks; nstage is a multiple of cwarps
  int tile_blocks;
  int cwarps;               // active consumer warps (<= K1_CWARPS)
};

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// TMA bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// same, with an L2 evict-first policy: the genotype matrix is streamed once and must not displace the background tables
__device__ __forceinline__ void bulk_g2s_stream(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// carry-save adder on 32 independent bit lanes: (hi, lo) = a + b + c
__device__ __forceinline__ void csa(uint32_t& hi, uint32_t& lo, uint32_t a, uint32_t b, uint32_t c) {
  const uint32_t l = a ^ b ^ c;                    // one LOP3 (0x96)
  const uint32_t h = (a & b) | (c & (a | b));      // one LOP3 (0xE8, majority)
  hi = h;
  lo = l;
}

// Bit-sliced population counter (Harley-Seal): total() = sum of popcounts of every word added.
struct BitCounter {
  uint32_t ones = 0, twos = 0, fours = 0, acc8 = 0;
  __device__ __forceinline__ void add8(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, uint32_t w4, uint32_t w5,
                                       uint32_t w6, uint32_t w7) {
    uint32_t t0, t1, t2, t3, f0, f1, e0;
    csa(t0, ones, ones, w0, w1);
    csa(t1, ones, ones, w2, w3);
    csa(t2, ones, ones, w4, w5);
    csa(t3, ones, ones, w6, w7);
    csa(f0, twos, twos, t0, t1);
    csa(f1, twos, twos, t2, t3);
    csa(e0, fours, fours, f0, f1);
    acc8 += __popc(e0);
  }
  __device__ __forceinline__ void add4(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
    uint32_t t0, t1, f0;
    csa(t0, ones, ones, w0, w1);
    csa(t1, ones, ones, w2, w3);
    csa(f0, twos, twos, t0, t1);
    uint32_t c = fours & f0;
    fours ^= f0;
    acc8 += __popc(c);
  }
  __device__ __forceinline__ void add2(uint32_t w0, uint32_t w1) {
    uint32_t t0;
    csa(t0, ones, ones, w0, w1);
    uint32_t c = twos & t0;
    twos ^= t0;
    uint32_t c2 = fours & c;
    fours ^= c;
    acc8 += __popc(c2);
  }
  __device__ __forceinline__ uint32_t total() const {
    return 8u * acc8 + 4u * __popc(fours) + 2u * __popc(twos) + __popc(ones);
  }
};

// MISSING plane of 32 samples from their two bit-plane words: code 0b10 = missing -> hi & ~lo (one LOP3).
__device__ __forceinline__ uint32_t missing_plane(uint32_t lo, uint32_t hi) { return hi & ~lo; }

// Per-population accumulation over one row block held in shared memory.
// Words come in (lo plane, hi plane) pairs of 32 samples.
// alt = popcount(all bits) - #missing   (codes 00 -> 0, 01 -> 1, 11 -> 2, 10 = missing -> popcount 1, removed)
struct PopCounts {
  BitCounter bits, miss;
  __device__ __forceinline__ void chunk4(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
    bits.add4(w0, w1, w2, w3);
    miss.add2(missing_plane(w0, w1), missing_plane(w2, w3));
  }
  __device__ __forceinline__ void chunk8(uint4 a, uint4 b) {
    bits.add8(a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w);
    miss.add4(missing_plane(a.x, a.y), missing_plane(a.z, a.w), missing_plane(b.x, b.y), missing_plane(b.z, b.w));
  }
};

// One population block of one SNP in the B32 layout: word w of the lane's SNP sits at blk[w * 32] (conflict-free LDS.32,
// immediate offsets after unrolling).  Returns T = popcount of all bits, M = number of missing calls.
template <int TW>  // TW > 0: compile-time word count (fully unrolled, immediate offsets); TW == 0: runtime W
__device__ __forceinline__ void count_block_b32(const uint32_t* blk, int Wrt, uint32_t& T, uint32_t& M) {
  const int W = TW > 0 ? TW : Wrt;
  PopCounts pc;
  int w = 0;
#pragma unroll
  for (; w + 8 <= W; w += 8) {
    const uint32_t* q = blk + w * BLK;
    uint4 a = make_uint4(q[0], q[BLK], q[2 * BLK], q[3 * BLK]);
    uint4 b = make_uint4(q[4 * BLK], q[5 * BLK], q[6 * BLK], q[7 * BLK]);
    pc.chunk8(a, b);
  }
  if (w + 4 <= W) {
    const uint32_t* q = blk + w * BLK;
    pc.chunk4(q[0], q[BLK], q[2 * BLK], q[3 * BLK]);
    w += 4;
  }
  if (w < W) {
    const uint32_t* q = blk + w * BLK;
    const uint32_t w0 = q[0];
    const uint32_t w1 = (w + 1 < W) ? q[BLK] : 0u;
    const uint32_t w2 = (w + 2 < W) ? q[2 * BLK] : 0u;
    pc.chunk4(w0, w1, w2, 0u);
  }
  T = pc.bits.total();
  M = pc.miss.total();
}

// ------------------------------------------------------------------------------------------------ row sink
// Shared-memory privatised background histograms of ONE background group per CTA.
struct SinkSmem {
  uint32_t* corner;  // [cr*cc]
  uint32_t* h1a;     // [h1a]
  uint32_t* h1b;     // [h1b]
};

struct ChromCache {
  int c = -1;
  long long lo = 0, hi = -1;
};

__device__ __forceinline__ int chrom_of_row(const KeyParams& p, long long s, ChromCache& cc) {
  if (s >= cc.lo && s < cc.hi) return cc.c;
  int lo = 0, hi = p.C;  // find c with off[c] <= s < off[c+1]
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (__ldg(p.chrom_off + mid) <= s) lo = mid; else hi = mid;
  }
  cc.c = lo;
  cc.lo = __ldg(p.chrom_off + lo);
  cc.hi = __ldg(p.chrom_off + lo + 1);
  return lo;
}

__device__ __forceinline__ int group_of_row(const KeyParams& p, long long s, ChromCache& cc) {
  int g = p.uniform_group;
  if (p.bg_group) g = __ldg(p.bg_group + chrom_of_row(p, s, cc));
  if (g >= 0 && p.bg_lo >= 0) {
    long long q = __ldg(p.pos + s);
    if (q < p.bg_lo || q > p.bg_hi) g = -1;
  }
  return g;
}

// 1D helper: folded bin of a raw alt count, 0 when the SNP does not enter the 1D likelihood
// (alt == 0 skipped :430; folded bins 0 and n dropped :488)
__device__ __forceinline__ int folded_interior(int a, int n) {
  int f = min(a, 2 * n - a);
  return (a != 0 && f >= 1 && f <= n - 1) ? f : 0;
}

// narrow record -> (2D bin, fa | fb << 16)
__device__ __forceinline__ uint2 decode_narrow(uint32_t r, const RecFmt& f, int n1, int n2, int C2) {
  const int k1 = (int)(r & ((1u << f.b1) - 1u)), k2 = (int)((r >> f.b1) & ((1u << f.b2) - 1u));
  const int d1 = (int)((r >> (f.b1 + f.b2)) & ((1u << f.md) - 1u)), d2 = (int)(r >> (f.b1 + f.b2 + f.md));
  return make_uint2((uint32_t)(k1 * C2 + k2),
                    (uint32_t)folded_interior(k1 + 2 * d1, n1) | ((uint32_t)folded_interior(k2 + 2 * d2, n2) << 16));
}
// record s of either format as (2D bin, fa | fb << 16); streamed (read once per pass)
__device__ __forceinline__ uint2 load_rec(const void* rec, const RecFmt& f, long long s, int n1, int n2, int C2) {
  if (f.narrow) return decode_narrow(__ldcs(reinterpret_cast<const uint32_t*>(rec) + s), f, n1, n2, C2);
  return __ldcs(reinterpret_cast<const uint2*>(rec) + s);
}

// snp_flags handling shared by the count kernels: returns whether the SNP passes the spectrum filters (bit0) and
// applies the sparse half-call corrections of rows flagged with bit2 (binary search in the sorted fix-up list).
__device__ __forceinline__ bool row_filters(const KeyParams& p, long long s, int& ref1, int& alt1, int& ref2, int& alt2) {
  if (!p.flags) return true;
  const uint8_t f = __ldg(p.flags + s);
  if (f & 4) {
    long long lo = 0, hi = p.nfix;
    while (lo < hi) {
      long long mid = (lo + hi) >> 1;
      if (p.fix[mid].snp < s) lo = mid + 1; else hi = mid;
    }
    for (; lo < p.nfix && p.fix[lo].snp == s; ++lo) {
      if (p.fix[lo].pop == 0) { ref1 += p.fix[lo].dref; alt1 += p.fix[lo].dalt; }
      else { ref2 += p.fix[lo].dref; alt2 += p.fix[lo].dalt; }
    }
  }
  return (f & 1) != 0;
}

// From the four counts of a SNP to its keys, the output arrays and the background histograms.  Returns (2D bin, fa | fb << 16).
__device__ __forceinline__ uint2 sink_row(const KeyParams& p, long long s, int ref1, int alt1, int ref2, int alt2, int cta_group,
                                          const SinkSmem& sm, ChromCache& cc) {
  const bool include = row_filters(p, s, ref1, alt1, ref2, alt2);
  uint32_t key = 0, alts = 0, nrec = 0;
  if (include) {
    int k1 = alt1, k2 = alt2;
    const bool swapped = p.fold && alt1 + alt2 > p.n1 + p.n2;
    if (swapped) { k1 = ref1; k2 = ref2; }  // twoDSFS_class.py:199-206
    if ((unsigned)k1 >= (unsigned)p.R1 || (unsigned)k2 >= (unsigned)p.R2 || (unsigned)alt1 >= (unsigned)p.R1 ||
        (unsigned)alt2 >= (unsigned)p.R2) {
      atomicOr(p.err, 1);
    } else {
      key = (uint32_t)(k1 * p.C2 + k2);  // (0,0) -> 0 : skipped SNP (:212)
      alts = (uint32_t)folded_interior(alt1, p.n1) | ((uint32_t)folded_interior(alt2, p.n2) << 16);
      if (p.fmt.narrow) {
        int d1 = 0, d2 = 0;
        if (swapped) {
          const int g1 = 2 * p.n1 - alt1 - ref1, g2 = 2 * p.n2 - alt2 - ref2;  // twice the missing diploids
          d1 = g1 >> 1; d2 = g2 >> 1;
          if (((g1 | g2) & 1) || g1 < 0 || g2 < 0 || d1 >= (1 << p.fmt.md) || d2 >= (1 << p.fmt.md)) {
            atomicOr(p.err, 8);  // does not fit the narrow record: the host redoes the pass with wide records
            d1 = d2 = 0;
          }
        }
        nrec = (uint32_t)k1 | ((uint32_t)k2 << p.fmt.b1) | ((uint32_t)d1 << (p.fmt.b1 + p.fmt.b2)) |
               ((uint32_t)d2 << (p.fmt.b1 + p.fmt.b2 + p.fmt.md));
      }
      const int g = group_of_row(p, s, cc);
      if (g >= 0) {
        uint32_t* gh = p.hist + (long long)g * p.gstride;
        if (key) {
          if (g == cta_group && k1 < p.cr && k2 < p.cc) atomicAdd(sm.corner + k1 * p.cc + k2, 1u);
          else atomicAdd(gh + key, 1u);
        }
        if (alt1) {
          if (g == cta_group && alt1 < p.h1a) atomicAdd(sm.h1a + alt1, 1u);
          else atomicAdd(gh + p.bins2d + alt1, 1u);
        }
        if (alt2) {
          if (g == cta_group && alt2 < p.h1b) atomicAdd(sm.h1b + alt2, 1u);
          else atomicAdd(gh + p.bins2d + p.R1 + alt2, 1u);
        }
      }
    }
  }
  // streaming store: read once by the scorer, from L2 or HBM
  if (p.fmt.narrow) __stcs(reinterpret_cast<uint32_t*>(p.rec) + s, nrec);
  else __stcs(reinterpret_cast<uint2*>(p.rec) + s, make_uint2(key, alts));
  return make_uint2(key, alts);
}

// flush the CTA-private histograms of group g into global memory (threads tid..nthr of the sink group)
__device__ __forceinline__ void sink_flush(const KeyParams& p, const SinkSmem& sm, int g, int tid, int nthr) {
  if (g < 0) return;
  uint32_t* gh = p.hist + (long long)g * p.gstride;
  for (int i = tid; i < p.cr * p.cc; i += nthr) {
    uint32_t v = sm.corner[i];
    if (v) {
      atomicAdd(gh + (i / p.cc) * p.C2 + (i % p.cc), v);
      sm.corner[i] = 0;
    }
  }
  for (int i = tid; i < p.h1a; i += nthr) {
    uint32_t v = sm.h1a[i];
    if (v) { atomicAdd(gh + p.bins2d + i, v); sm.h1a[i] = 0; }
  }
  for (int i = tid; i < p.h1b; i += nthr) {
    uint32_t v = sm.h1b[i];
    if (v) { atomicAdd(gh + p.bins2d + p.R1 + i, v); sm.h1b[i] = 0; }
  }
}

__device__ __forceinline__ int tile_group(const KeyParams& p, long long row0, ChromCache& cc) {
  if (!p.bg_group) return p.uniform_group;
  return __ldg(p.bg_group + chrom_of_row(p, row0, cc));
}

// ------------------------------------------------------------------------------------------------ K1 (genotypes)
// K1 for rows wider than one stage of k1_fused's ring (more than 4096 samples): a 32-SNP block is streamed as segments of
// `seg_words` words (contiguous in the B32 layout); the warp carries its bit-sliced counters across the segments of a block
// and sinks the SNPs after the last one.  Generic (runtime) geometry: the population of a word is decided per segment piece.
__global__ void __launch_bounds__(K1_THREADS, 1) k1_genotypes_wide(const __grid_constant__ KeyParams p, int seg_words) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int W1 = p.W1, W2 = p.W2, RW = W1 + W2;
  const int nseg = (RW + seg_words - 1) / seg_words;
  uint8_t* stages = smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)p.nstage * p.stage_bytes);
  SinkSmem sm;
  sm.corner = reinterpret_cast<uint32_t*>(full + p.nstage);
  sm.h1a = sm.corner + p.cr * p.cc;
  sm.h1b = sm.h1a + p.h1a;
  const int nhist = p.cr * p.cc + p.h1a + p.h1b;
  if (tid == 0) {
    for (int i = 0; i < p.nstage; ++i) mbar_init(full + i, 1);
    fence_barrier_init();
  }
  for (int i = tid; i < nhist; i += blockDim.x) sm.corner[i] = 0;
  __syncthreads();
  const long long b0 = p.r0 / BLK, b1 = (p.r1 + BLK - 1) / BLK;
  const long long nblk = b1 - b0;
  const long long t0 = nblk * blockIdx.x / gridDim.x, t1 = nblk * (blockIdx.x + 1) / gridDim.x;
  const long long block_words = (long long)RW * BLK;
  const int depth = p.nstage / p.cwarps;
  ChromCache cc;
  const int cta_group = (t1 > t0) ? tile_group(p, p.r0 + t0 * BLK, cc) : -1;
  if (warp < p.cwarps) {
    uint8_t* my_stages = stages + (size_t)warp * depth * p.stage_bytes;
    uint64_t* my_full = full + warp * depth;
    // warp w owns blocks t0 + w, t0 + w + cwarps, ...; its item j = (own block j / nseg, segment j % nseg)
    const long long my_blocks = (t1 - t0 > warp) ? (t1 - t0 - warp + p.cwarps - 1) / p.cwarps : 0;
    const long long my_items = my_blocks * nseg;
    auto issue = [&](long long j, int slot) {  // lane 0 only
      const long long blk = b0 + t0 + warp + (j / nseg) * p.cwarps;
      const int sg = (int)(j % nseg);
      const int w0 = sg * seg_words, nw = min(seg_words, RW - w0);
      const uint32_t bytes = (uint32_t)nw * BLK * 4;
      mbar_arrive_expect_tx(my_full + slot, bytes);
      bulk_g2s_stream(my_stages + (size_t)slot * p.stage_bytes, p.G + blk * block_words + (long long)w0 * BLK, bytes, my_full + slot);
    };
    if (lane == 0)
      for (int j = 0; j < depth && j < my_items; ++j) issue(j, j);
    int slot = 0;
    uint32_t ph = 0;
    PopCounts pc1, pc2;
    for (long long j = 0; j < my_items; ++j) {
      const int sg = (int)(j % nseg);
      const int w0 = sg * seg_words, nw = min(seg_words, RW - w0);
      mbar_wait(my_full + slot, ph);
      const uint32_t* q = reinterpret_cast<const uint32_t*>(my_stages + (size_t)slot * p.stage_bytes) + lane;
      // words [w0, w0+nw): the part below W1 belongs to population 1, the rest to population 2
      const int n1w = max(0, min(nw, W1 - w0));
      for (int w = 0; w < n1w; w += 4)
        pc1.chunk4(q[w * BLK], w + 1 < n1w ? q[(w + 1) * BLK] : 0u, w + 2 < n1w ? q[(w + 2) * BLK] : 0u, w + 3 < n1w ? q[(w + 3) * BLK] : 0u);
      for (int w = n1w; w < nw; w += 4)
        pc2.chunk4(q[w * BLK], w + 1 < nw ? q[(w + 1) * BLK] : 0u, w + 2 < nw ? q[(w + 2) * BLK] : 0u, w + 3 < nw ? q[(w + 3) * BLK] : 0u);
      __syncwarp();
      if (lane == 0 && j + depth < my_items) {
        fence_proxy_async();
        issue(j + depth, slot);
      }
      if (++slot == depth) { slot = 0; ph ^= 1; }
      if (sg == nseg - 1) {  // last segment of the block: sink its 32 SNPs
        const long long s = (b0 + t0 + warp + (j / nseg) * p.cwarps) * BLK + lane;
        if (s < p.r1) {
          const uint32_t T1 = pc1.bits.total(), M1 = pc1.miss.total(), T2 = pc2.bits.total(), M2 = pc2.miss.total();
          const int alt1 = (int)(T1 - M1), alt2 = (int)(T2 - M2);
          const int ref1 = 2 * (p.ns1 - (int)M1) - alt1, ref2 = 2 * (p.ns2 - (int)M2) - alt2;
          sink_row(p, s, ref1, alt1, ref2, alt2, cta_group, sm, cc);
        }
        pc1 = PopCounts();
        pc2 = PopCounts();
      }
    }
  }
  __syncthreads();
  sink_flush(p, sm, cta_group, tid, blockDim.x);
}

// ------------------------------------------------------------------------------------------------ peer exchange
// In-place all-reduce (sum) of the packed background histogram over the GPUs of one NVSwitch node, through peer memory
// (CUDA IPC mappings of every rank's histogram): rank r pulls slice r of every rank, sums it and pushes the sum back
// into slice r of every rank.  Ranks meet at a flag barrier before (all count kernels finished) and after (all pushes
// landed).  flags[q][r] on rank q holds the last epoch rank r signalled.
constexpr int PEER_MAX = 16;
struct PeerParams {
  uint32_t* hist[PEER_MAX];
  unsigned long long* flags[PEER_MAX];
  int rank, world;
  long long words;
  int* err;
  long long timeout_cycles;
  unsigned int* ticket;      // CTA arrival counter of peer_exchange (reset by its last CTA)
};

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// spin until the flag (in THIS rank's memory, written by a peer) reaches `epoch`; a peer that never arrives flags an error
__device__ __forceinline__ void peer_wait(const unsigned long long* flag, unsigned long long epoch, int* err, long long timeout_cycles) {
  const long long t0 = clock64();
  while (ld_acquire_sys(flag) < epoch) {
    if (clock64() - t0 > timeout_cycles) {
      atomicOr(err, 4);
      break;
    }
  }
}

// ------------------------------------------------------------------------------------------------ K1 (counts entry)
constexpr int K1C_THREADS = 256;
__global__ void __launch_bounds__(K1C_THREADS) k1_counts(const __grid_constant__ KeyParams p) {
  extern __shared__ __align__(16) uint8_t smem_c[];
  SinkSmem sm;
  sm.corner = reinterpret_cast<uint32_t*>(smem_c);
  sm.h1a = sm.corner + p.cr * p.cc;
  sm.h1b = sm.h1a + p.h1a;
  const int nhist = p.cr * p.cc + p.h1a + p.h1b;
  const int tid = threadIdx.x;
  for (int i = tid; i < nhist; i += K1C_THREADS) sm.corner[i] = 0;
  __syncthreads();
  const long long ntiles = (p.r1 - p.r0 + K1C_THREADS - 1) / K1C_THREADS;
  const long long t0 = ntiles * blockIdx.x / gridDim.x;
  const long long t1 = ntiles * (blockIdx.x + 1) / gridDim.x;
  ChromCache cc;
  int cta_group = -2;
  for (long long t = t0; t < t1; ++t) {
    const long long row0 = p.r0 + t * K1C_THREADS;
    const long long s = row0 + tid;
    const int g0 = tile_group(p, row0, cc);
    if (g0 != cta_group) {  // uniform across the CTA: switch the privatised histograms to the new background group
      __syncthreads();
      sink_flush(p, sm, cta_group, tid, K1C_THREADS);
      __syncthreads();
      cta_group = g0;
    }
    if (s < p.r1) {
      const uint2 v = __ldg(reinterpret_cast<const uint2*>(p.cnt) + s);  // (ref1 | alt1<<16, ref2 | alt2<<16)
      sink_row(p, s, (int)(v.x & 0xFFFF), (int)(v.x >> 16), (int)(v.y & 0xFFFF), (int)(v.y >> 16), cta_group, sm, cc);
    }
  }
  __syncthreads();
  sink_flush(p, sm, cta_group, tid, K1C_THREADS);
}

// ------------------------------------------------------------------------------------------------ background finalize
// ln b_k tables and interior totals B from the integer histograms (fold_1d_sfs :446-463 applied here).
struct FinParams {
  const uint32_t* hist;
  long long gstride;
  int NG, bins2d, R1, R2, n1, n2;
  double* lb2;   // [NG][bins2d]
  double* lb1a;  // [NG][n1+1]
  double* lb1b;  // [NG][n2+1]
  unsigned long long* Bsum;  // [NG][3] interior totals, then one word used as the CTA arrival counter; zero between launches
  double* B;                 // [NG][6] = B (2D, 1D pop1, 1D pop2) then ln B
};

__device__ __forceinline__ double ln_count(unsigned long long v) { return v ? log((double)v) : -INFINITY; }

// ln tables and interior totals of background group g, by CTA `cta` of the `ncta` CTAs that share the group
__device__ __forceinline__ void finalize_tables(const FinParams& p, int g, int cta, int ncta) {
  const uint32_t* h = p.hist + (long long)g * p.gstride;
  unsigned long long local = 0;
  // four bins per thread and round, their loads issued together (in the count kernel's tail a thread has ~15 bins of a 1 M-bin
  // spectrum, and a load per iteration made the loop a chain of L2 latencies: 9 us -> 6.5 us; eight per round with predicated
  // slots measured no better than one)
  constexpr int U = 4;
  const long long stride = (long long)ncta * blockDim.x;
  double* lb2 = p.lb2 + (long long)g * p.bins2d;
  long long k = (long long)cta * blockDim.x + threadIdx.x;
  for (; k + (U - 1) * stride < p.bins2d; k += U * stride) {
    uint32_t v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = __ldcg(h + k + u * stride);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long kk = k + u * stride;
      lb2[kk] = ln_count(v[u]);
      if (kk > 0 && kk < p.bins2d - 1) local += v[u];
    }
  }
  for (; k < p.bins2d; k += stride) {
    const uint32_t v = __ldcg(h + k);
    lb2[k] = ln_count(v);
    if (k > 0 && k < p.bins2d - 1) local += v;
  }
  for (int o = 16; o; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(p.Bsum + g * 3, local);
  if (cta == 0) {
    for (int pop = 0; pop < 2; ++pop) {
      const int n = pop ? p.n2 : p.n1;
      const uint32_t* raw = h + p.bins2d + (pop ? p.R1 : 0);
      double* lb = pop ? p.lb1b + (long long)g * (p.n2 + 1) : p.lb1a + (long long)g * (p.n1 + 1);
      unsigned long long loc = 0;
      for (int k = threadIdx.x; k <= n; k += blockDim.x) {
        unsigned long long v = raw[k];
        if (2 * n - k != k) v += raw[2 * n - k];
        lb[k] = ln_count(v);
        if (k >= 1 && k <= n - 1) loc += v;
      }
      for (int o = 16; o; o >>= 1) loc += __shfl_xor_sync(0xffffffffu, loc, o);
      if ((threadIdx.x & 31) == 0 && loc) atomicAdd(p.Bsum + g * 3 + 1 + pop, loc);
    }
  }
}

// every CTA that ran finalize_tables calls this once afterwards: the last one to arrive turns the interior totals of all groups
// into the table [group][6] = B then ln B, and re-zeroes the sums
__device__ __forceinline__ void finalize_totals(const FinParams& p, int ctas_total) {
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  unsigned int* ticket = reinterpret_cast<unsigned int*>(p.Bsum + (long long)p.NG * 3);
  if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == (unsigned)ctas_total - 1;
  __syncthreads();
  if (s_last) {
    __threadfence();
    for (int i = threadIdx.x; i < p.NG * 3; i += blockDim.x) {
      const double b = (double)atomicExch(p.Bsum + i, 0ull);
      p.B[(i / 3) * 6 + i % 3] = b;
      p.B[(i / 3) * 6 + 3 + i % 3] = b > 0.0 ? log(b) : -INFINITY;
    }
    if (threadIdx.x == 0) *ticket = 0;
  }
}

__global__ void __launch_bounds__(256) k_finalize_counts(const __grid_constant__ FinParams p) {
  finalize_tables(p, blockIdx.y, blockIdx.x, gridDim.x);
  finalize_totals(p, gridDim.x * gridDim.y);
}

// Multi-GPU, ONE launch per rank between the count kernel and the finish kernel: [barrier: every rank's count kernel is
// done] -> pull slice `rank` of every rank's histogram over NVLink, sum, push the sum into every rank's histogram ->
// [barrier: every rank's pushes have landed] -> ln tables and totals of the (now complete) local histogram.  The epoch of
// the flag barriers lives in device memory (words[0] of `epoch_mem`, advanced by 2 by the last CTA) so that the launch can be
// replayed unchanged.  Grid <= number of SMs: every CTA is resident while it spins on the flags.
struct PeerFinParams {
  PeerParams x;
  FinParams f;
  unsigned long long* epoch_mem;  // [0] = last epoch used on this rank
};

// the exchange proper, by every CTA of a launch whose CTAs are all resident (they spin on the flags)
// `stamps` (diagnostics, normally null): CTA 0 leaves clock64 after barrier 1 [3], after its pushes are fenced [4] and after
// barrier 2 [5]
// No wait is needed after the launch: it returns only once every rank has signalled e + 1, and a rank signals only after it
// has read its slice from every histogram, summed it, pushed the sum and fenced (__threadfence_system).  So when the launch
// ends no peer still reads or writes this rank's histogram, and the next count kernel may zero and refill it.
__device__ __forceinline__ void peer_exchange(const PeerParams& p, unsigned long long* epoch_mem, unsigned long long* stamps = nullptr) {
  __shared__ int s_last2;
  auto stamp = [&](int i) { if (stamps && blockIdx.x == 0 && threadIdx.x == 0) stamps[i] = (unsigned long long)clock64(); };
  const unsigned long long e = *reinterpret_cast<volatile unsigned long long*>(epoch_mem) + 1;
  if ((int)threadIdx.x < p.world) {
    if (blockIdx.x == 0) {
      __threadfence_system();
      st_release_sys(p.flags[threadIdx.x] + p.rank, e);
    }
    peer_wait(p.flags[p.rank] + threadIdx.x, e, p.err, p.timeout_cycles);
  }
  __syncthreads();
  stamp(3);
  const long long n4 = p.words / 4;
  const long long lo = n4 * p.rank / p.world, hi = n4 * (p.rank + 1) / p.world;
  for (long long i = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (long long)gridDim.x * blockDim.x) {
    uint4 v[8];
#pragma unroll
    for (int r = 0; r < 8; ++r)
      if (r < p.world) v[r] = __ldcg(reinterpret_cast<const uint4*>(p.hist[r]) + i);
    uint4 s = make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int r = 0; r < 8; ++r)
      if (r < p.world) { s.x += v[r].x; s.y += v[r].y; s.z += v[r].z; s.w += v[r].w; }
    for (int r = 8; r < p.world; ++r) {
      const uint4 t = __ldcg(reinterpret_cast<const uint4*>(p.hist[r]) + i);
      s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
    }
    for (int r = 0; r < p.world; ++r) __stcg(reinterpret_cast<uint4*>(p.hist[r]) + i, s);
  }
  if (p.rank == p.world - 1 && blockIdx.x == 0 && threadIdx.x == 0)
    for (long long w = n4 * 4; w < p.words; ++w) {
      uint32_t s = 0;
      for (int r = 0; r < p.world; ++r) s += __ldcg(p.hist[r] + w);
      for (int r = 0; r < p.world; ++r) __stcg(p.hist[r] + w, s);
    }
  // every thread's pushes are ordered before the CTA's ticket; the last CTA tells every rank that this rank is done
  __threadfence_system();
  __syncthreads();
  stamp(4);
  if (threadIdx.x == 0) s_last2 = atomicAdd(p.ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last2 && (int)threadIdx.x < p.world) {
    __threadfence_system();
    st_release_sys(p.flags[threadIdx.x] + p.rank, e + 1);
  }
  // second barrier: every rank's slice has landed in this rank's histogram
  if ((int)threadIdx.x < p.world) peer_wait(p.flags[p.rank] + threadIdx.x, e + 1, p.err, p.timeout_cycles);
  __syncthreads();
  stamp(5);
  // every CTA has arrived at the ticket, so all of them read the epoch long ago: the last one advances it and resets the ticket
  if (s_last2 && threadIdx.x == 0) {
    *p.ticket = 0;
    *epoch_mem = e + 1;
  }
}

__global__ void __launch_bounds__(256) k_peer_reduce_finalize(const __grid_constant__ PeerFinParams q) {
  peer_exchange(q.x, q.epoch_mem);
  finalize_tables(q.f, 0, blockIdx.x, gridDim.x);
  finalize_totals(q.f, gridDim.x);
}

// Grid-wide barrier for launches whose CTAs are all resident (at most one CTA per SM): sense reversing, so the launch can be
// replayed without resetting anything.  bar[0] = arrivals, bar[1] = phase.  A CTA that never arrives flags error bit 4 after
// the timeout instead of hanging the others.
__device__ __forceinline__ void grid_barrier(unsigned int* bar, int* err, long long timeout_cycles) {
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    volatile unsigned int* phase = bar + 1;
    const unsigned int old = *phase;  // read before arriving: the phase cannot advance without this CTA
    if (atomicAdd(bar, 1u) == gridDim.x - 1) {
      *bar = 0;
      __threadfence();
      atomicAdd(bar + 1, 1u);
    } else {
      const long long t0 = clock64();
      while (*phase == old) {
        if (clock64() - t0 > timeout_cycles) {
          atomicOr(err, 16);
          break;
        }
      }
    }
    __threadfence();
  }
  __syncthreads();
}

// precomputed (float) background: lb = ln b
__global__ void k_log_table(const double* b, double* lb, long long n) {
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
    const double v = b[k];
    lb[k] = v > 0.0 ? log(v) : (v == 0.0 ? -INFINITY : NAN);
  }
}

__global__ void k_ln_int_table(double* t, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) t[i] = i ? log((double)i) : 0.0;
}

// ------------------------------------------------------------------------------------------------ K2 boundaries
struct WinParams {
  const int32_t* pos;
  const long long* chrom_off;
  const long long* cand_off;  // [C+1] candidate offsets per chromosome
  int C;
  long long W;                // window size in bp (fixed-bp) or SNPs (fixed-SNP)
  long long ncand;
  int32_t* wlo;
  int32_t* whi;
  int32_t* wchrom;
  long long* wstart;
  long long* wend;
  int32_t* large;             // ids of windows with more than `wcap` SNPs
  int* nlarge;
  int32_t* r_count;           // result arrays: K2 marks empty candidates itself
  uint8_t* r_flags;
  int wcap;                   // WCAP, or 0 when the panel is too large for the shared-memory scorer (every window "large")
};

__device__ __forceinline__ long long lower_bound_pos(const int32_t* pos, long long lo, long long hi, long long v) {
  while (lo < hi) {
    long long mid = (lo + hi) >> 1;
    if ((long long)__ldg(pos + mid) < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ int cand_chrom(const WinParams& p, long long id) {
  int lo = 0, hi = p.C;
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (__ldg(p.cand_off + mid) <= id) lo = mid; else hi = mid;
  }
  return lo;
}

// fixed-bp: window k of a chromosome holds positions [1+kW, (k+1)W]; position 0 falls in window 0 (:898, Q10)
__global__ void __launch_bounds__(256) k2_bounds_bp(const __grid_constant__ WinParams p) {
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= p.ncand) return;
  const int c = cand_chrom(p, id);
  const long long k = id - __ldg(p.cand_off + c);
  const long long clo = __ldg(p.chrom_off + c), chi = __ldg(p.chrom_off + c + 1);
  const long long lo = k == 0 ? clo : lower_bound_pos(p.pos, clo, chi, 1 + k * p.W);
  const long long hi = lower_bound_pos(p.pos, lo, chi, 1 + (k + 1) * p.W);
  p.wlo[id] = (int32_t)lo;
  p.whi[id] = (int32_t)hi;
  p.wchrom[id] = c;
  if (hi == lo) { p.r_count[id] = 0; p.r_flags[id] = TDSFS_F_EMPTY; }  // the reference never emits an empty window
  p.wstart[id] = 1 + k * p.W;
  p.wend[id] = (k + 1) * p.W;
  if (hi - lo > p.wcap) p.large[atomicAdd(p.nlarge, 1)] = (int32_t)id;
}

// fixed-SNP: chunk j of a chromosome = rows [off + jN, off + (j+1)N); label per :1527/:1535
__global__ void __launch_bounds__(256) k2_bounds_snp(const __grid_constant__ WinParams p) {
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= p.ncand) return;
  const int c = cand_chrom(p, id);
  const long long j = id - __ldg(p.cand_off + c);
  const long long lo = __ldg(p.chrom_off + c) + j * p.W, hi = lo + p.W;
  p.wlo[id] = (int32_t)lo;
  p.whi[id] = (int32_t)hi;
  p.wchrom[id] = c;
  p.wstart[id] = j == 0 ? (long long)__ldg(p.pos + lo) : (long long)__ldg(p.pos + lo - 1) + 1;
  p.wend[id] = (long long)__ldg(p.pos + hi - 1);
  if (hi - lo > p.wcap) p.large[atomicAdd(p.nlarge, 1)] = (int32_t)id;
}

// ------------------------------------------------------------------------------------------------ K3+K4 scoring
struct ScoreParams {
  const void* rec;       // per-SNP records (RecFmt)
  RecFmt fmt;
  int C2;                // 2 n2 + 1
  // legacy Poisson composite score (reference scripts/twoDSFS.py:336-463) instead of the likelihood ratios: lb2 holds ln q of
  // the normalised background (-inf where q = 0), the spectrum is unfolded and every bin but (0,0) counts
  int poisson;
  double pq_n, pq_sum, pq_lnsum;  // number of bins with q != 0, their sum, the sum of their logarithms
  const uint8_t* flags;
  const int32_t* wlo;
  const int32_t* whi;
  const int32_t* wchrom;
  const int32_t* score_group;  // per chromosome (NULL = group 0)
  long long ncand;
  int n1, n2, bins2d, snp_mode;
  // dynamic window assignment: a group takes window atomicAdd(work, 1) - work_base until that is >= ncand; every group
  // fails exactly once per launch, so the host advances work_base by ncand + groups and the counter never needs a reset
  unsigned long long* work;
  unsigned long long work_base;
  const double* lb2;
  const double* lb1a;
  const double* lb1b;
  const double* B;       // [NG][6]: interior totals B (2D, 1D pop1, 1D pop2), then ln B
  const double* lnI;     // ln(m), m < LN_TABLE
  // outputs
  int32_t* r_count;
  int32_t* r_n2;
  int32_t* r_n1a;
  int32_t* r_n1b;
  double* r_T2;
  double* r_T1a;
  double* r_T1b;
  uint8_t* r_flags;
  // large-window path
  const int32_t* large;
  const int* nlarge;
  uint32_t* scratch;     // [nCTA][bins2d + n1 + 1 + n2 + 1]
};

__device__ __forceinline__ double ln_mult(const ScoreParams& p, uint32_t m) {
  return m < (uint32_t)LN_TABLE ? __ldg(p.lnI + m) : log((double)m);
}

__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// T = 2 * ( sum_k x_k (ln x_k - ln b_k)  -  N (ln N - ln B) )   ==  2 (ll_fg - ll_bg) of the reference (:679-682)
// acc = sum_k x_k (ln x_k - ln b_k); Bg = {B[3], lnB[3]} of the background group; q = 0 (2D), 1, 2 (1D pops)
__device__ __forceinline__ double clr_value(const ScoreParams& p, int N, double acc, const double* Bg, int q, bool& none) {
  const double B = __ldg(Bg + q);
  none = (N == 0) || !(B != 0.0);  // the reference returns None (:645-647, :668-670)
  if (none) return NAN;
  // explicit roundings (no FMA contraction): a window whose only populated bin is the only background bin, or a window
  // that is its own background, must give exactly 0.0 like the reference -- its truthiness drives the stale-carry quirk
  const double t = __dsub_rn(ln_mult(p, (uint32_t)N), __ldg(Bg + 3 + q));
  return 2.0 * __dsub_rn(acc, __dmul_rn((double)N, t));
}

__device__ __forceinline__ void write_result(const ScoreParams& p, long long id, int count, int nall, int N2, int N1a, int N1b,
                                             double acc2, double acc1a, double acc1b, const double* Bg) {
  bool none2, none1a, none1b;
  const double T2 = clr_value(p, N2, acc2, Bg, 0, none2);
  const double T1a = clr_value(p, N1a, acc1a, Bg, 1, none1a);
  const double T1b = clr_value(p, N1b, acc1b, Bg, 2, none1b);
  uint8_t f = (none2 ? TDSFS_F_T2D_NONE : 0) | (none1a ? TDSFS_F_T1D_P1_NONE : 0) | (none1b ? TDSFS_F_T1D_P2_NONE : 0);
  if (p.snp_mode && nall == 0) f |= TDSFS_F_SKIPPED;  // :1496 window skipped when its 2D spectrum sums to 0
  p.r_count[id] = count;
  p.r_n2[id] = N2;
  p.r_n1a[id] = N1a;
  p.r_n1b[id] = N1b;
  p.r_T2[id] = T2;
  p.r_T1a[id] = T1a;
  p.r_T1b[id] = T1b;
  p.r_flags[id] = f;
}

// Legacy Poisson score of one window (reference :295-303, :346-371), for both scorers: the sum over the bins with q != 0 of
// poisson.logpmf(int(x + 1/total), S_w q), S_w = total + bins / total, from the window's sums over its populated bins with
// q != 0 (xq = sum x, xlnq = sum x ln q, lg0 / lg1 = sum lgamma(x + 1) / lgamma(x + 2)):
//   (e nQ + xq) ln S_w + e sum ln q + xlnq - S_w sum q - sum lgamma(x + e + 1),   e = 1 only when total == 1
// (int(x + 1/total) = x + e in every bin).  A window with no counted SNP scores 0: the reference's S_w is 0 then.
__device__ __forceinline__ double poisson_finish(const ScoreParams& p, int total, double xq, double xlnq, double lg0, double lg1) {
  if (total == 0) return 0.0;
  const double Sw = (double)total + (double)p.bins2d / (double)total;
  const double e = total == 1 ? 1.0 : 0.0;
  return (e * p.pq_n + xq) * log(Sw) + e * p.pq_lnsum + xlnq - Sw * p.pq_sum - (total == 1 ? lg1 : lg0);
}

// A group of G warps per candidate window (<= WCAP SNPs), 8 warps per CTA.  Per-group shared memory: an open-addressing
// table of the window's 2D bins (one word per slot: bin << 10 | multiplicity), the list of occupied slots, packed
// 16-bit folded 1D histograms and a small reduction scratch.
//   pass 1 (per SNP)          insert the 2D bin, bump the two folded 1D bins      (all records of a thread in flight)
//   pass 2 (table walk)       acc += x (ln x - ln b) for every occupied slot, cleared on the way
//   pass 3 (per 1D bin pair)  same for both 1D spectra, bins cleared on the way
// Several warps per window keep the same shared-memory footprint per window but multiply the resident warps, which is
// what hides the shared-atomic and gather latencies.
constexpr int SCORE_WARPS = 8;
constexpr int KEY_SHIFT = 10;  // multiplicity field (< 1024, WCAP = 768)
__host__ __device__ inline int score_group_smem_words(int n1, int n2) {
  // table | 1D bins (padded to an even word count) | reduction scratch (SCORE_WARPS x 10 words)
  return HASH_SLOTS + (((n1 + 2) / 2 + (n2 + 2) / 2 + 1) & ~1) + SCORE_WARPS * 10 + 2;
}
// limits of the shared-memory scorer; panels beyond them are scored by the CTA kernel only
__host__ __device__ inline bool score_small_ok(int n1, int n2, int bins2d) {
  return n1 <= 32767 && n2 <= 32767 && bins2d < (1 << (32 - KEY_SHIFT)) - 1;
}

// exact uint32 -> double on the integer + fp64 pipes (I2F.F64 runs on the quarter-rate conversion unit)
__device__ __forceinline__ double u32_to_double(uint32_t x) {
  return __hiloint2double(0x43300000, (int)x) - 4503599627370496.0;  // 2^52 + x, minus 2^52
}

// predicated shared-memory reduction (no branch, no return value): bump the 16-bit half `f & 1` of word `f >> 1` when f != 0
__device__ __forceinline__ void bump_half_if(uint32_t* h, uint32_t f) {
  const uint32_t addr = smem_u32(h) + ((f << 1) & ~3u);
  const uint32_t val = (f & 1u) ? 0x10000u : 1u;
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p red.shared.add.u32 [%1], %2;\n\t}" ::"r"(f), "r"(addr), "r"(val) : "memory");
}

// EXTRA = the scan has per-SNP flags or fixed-SNP windows (extra per-record bookkeeping); false for the plain fixed-bp scan
template <int G, bool EXTRA>
__global__ void __launch_bounds__(SCORE_WARPS * 32) k3_score_small(const __grid_constant__ ScoreParams p) {
  extern __shared__ __align__(16) uint32_t sm32[];
  constexpr int GT = G * 32;                 // threads per group (SCORE_WARPS / G groups per CTA)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int grp = warp / G, wg = warp % G, tg = wg * 32 + lane;
  const int gwords = score_group_smem_words(p.n1, p.n2);
  uint32_t* tab = sm32 + (size_t)grp * gwords;
  uint32_t* h1a = tab + HASH_SLOTS;            // packed 16-bit bins: bin f in word f >> 1, half f & 1
  const int nw1 = (p.n1 + 2) / 2, nw2 = (p.n2 + 2) / 2;
  uint32_t* h1b = h1a + nw1;
  uint32_t* red = h1a + ((nw1 + nw2 + 1) & ~1);  // [G][10] (8-byte aligned): per warp {a2, a1a, a1b (doubles), N-pack, count, nall}
  auto gsync = [&]() {
    if (G == 1) __syncwarp(); else named_bar_sync(1 + grp, GT);
  };
  for (int i = tg; i < HASH_SLOTS; i += GT) tab[i] = EMPTY_KEY;
  for (int i = tg; i < nw1 + nw2; i += GT) h1a[i] = 0;
  gsync();
  const uint32_t last = p.poisson ? 0xFFFFFFFFu : (uint32_t)p.bins2d - 1;
  const bool has_flags = EXTRA && p.flags != nullptr;
  const bool snp_mode = EXTRA && p.snp_mode;

  // windows are handed out dynamically (an atomic counter): with a few windows per warp a static round-robin leaves
  // most warps idle while the ones that drew one window more finish
  auto grab = [&]() -> long long {
    long long v = 0;
    if (G == 1) {
      if (lane == 0) v = (long long)(atomicAdd(p.work, 1ull) - p.work_base);
      v = __shfl_sync(0xffffffffu, v, 0);
    } else {
      volatile long long* slot = reinterpret_cast<volatile long long*>(red + SCORE_WARPS * 10);
      if (tg == 0) *slot = (long long)(atomicAdd(p.work, 1ull) - p.work_base);
      gsync();
      v = *slot;
      gsync();
    }
    return v;
  };
  for (long long id = grab(); id < p.ncand; id = grab()) {
    const int lo = __ldg(p.wlo + id), hi = __ldg(p.whi + id);
    const int cnt = hi - lo;
    if (cnt == 0) {
      if (tg == 0) { p.r_count[id] = 0; p.r_flags[id] = TDSFS_F_EMPTY; }
      continue;
    }
    if (cnt > WCAP) continue;  // scored by k3_score_large
    const int g = p.score_group ? __ldg(p.score_group + __ldg(p.wchrom + id)) : 0;
    const double* lb2 = p.lb2 + (long long)g * p.bins2d;
    const double* lb1a = p.lb1a + (long long)g * (p.n1 + 1);
    const double* lb1b = p.lb1b + (long long)g * (p.n2 + 1);

    // ---- pass 1: up to Q records per thread in flight (the loads are independent of the table work)
    constexpr int Q = G == 1 ? 8 : 4;
    int count = 0, nall = 0;
    for (int base = 0; base < cnt; base += Q * GT) {
      uint2 r[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int i = base + q * GT + tg;
        r[q] = i < cnt ? load_rec(p.rec, p.fmt, lo + i, p.n1, p.n2, p.C2) : make_uint2(0u, 0u);  // streamed once: keep the ln b table in L2
        if (has_flags && i < cnt) count += (__ldg(p.flags + lo + i) >> 1) & 1;
      }
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const uint32_t k = r[q].x;
        if (snp_mode) nall += k != 0;
        if (k != 0 && k != last) {
          uint32_t h = (k * 0x9E3779B1u) >> 22;  // HASH_SLOTS = 2^10
          while (true) {  // read first: a shared-memory CAS costs about twice a load or an add
            uint32_t e = tab[h];
            if (e == EMPTY_KEY) {
              e = atomicCAS(tab + h, EMPTY_KEY, (k << KEY_SHIFT) | 1u);
              if (e == EMPTY_KEY) break;
            }
            if ((e >> KEY_SHIFT) == k) { atomicAdd(tab + h, 1u); break; }
            h = (h + 1) & (HASH_SLOTS - 1);
          }
        }
        const uint32_t fa = r[q].y & 0xFFFF, fb = r[q].y >> 16;
        bump_half_if(h1a, fa);
        bump_half_if(h1b, fb);
      }
    }
    gsync();
    // ---- pass 2: walk the table (shared-memory atomics are the scarce resource here: no occupied-slot list is kept).
    // U slots per thread are read first and all their ln b / ln x gathers issued together, branch-free: the gathers
    // come from L2 (~700 cycles), so their number in flight - not their count - sets the time of this pass.
    double a2 = 0.0, a1a = 0.0, a1b = 0.0;
    uint32_t N2 = 0, N1a = 0, N1b = 0;
    double pz_lg0 = 0.0, pz_lg1 = 0.0;  // Poisson score: sum of lgamma(x + 1) and of lgamma(x + 2) over the bins with q != 0
    uint32_t pz_xq = 0;                 // ... and the number of SNPs in those bins
    if (EXTRA && p.poisson) {
      // the table walk of the Poisson score: x ln q - lgamma(x + 1) over the populated bins with a non-zero expectation
      for (int j0 = tg; j0 < HASH_SLOTS; j0 += GT) {
        const uint32_t e = tab[j0];
        if (e != EMPTY_KEY) {
          tab[j0] = EMPTY_KEY;
          const uint32_t x = e & ((1u << KEY_SHIFT) - 1);
          const double lq = __ldg(lb2 + (e >> KEY_SHIFT));
          N2 += x;
          if (lq != -INFINITY) {  // a zero expectation is skipped (:364)
            a2 = fma(u32_to_double(x), lq, a2);
            pz_lg0 += lgamma((double)x + 1.0);
            pz_lg1 += lgamma((double)x + 2.0);
            pz_xq += x;
          }
        }
      }
    } else {
      constexpr int PER = HASH_SLOTS / GT;       // slots per thread
      constexpr int U = PER < 8 ? PER : 8;
#pragma unroll 1
      for (int j0 = tg; j0 < HASH_SLOTS; j0 += U * GT) {
        uint32_t e[U];
        double lbv[U], lnx[U];
#pragma unroll
        for (int u = 0; u < U; ++u) e[u] = tab[j0 + u * GT];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const bool occ = e[u] != EMPTY_KEY;
          const uint32_t x = occ ? (e[u] & ((1u << KEY_SHIFT) - 1)) : 0u;
          lbv[u] = occ ? __ldg(lb2 + (e[u] >> KEY_SHIFT)) : 0.0;
          lnx[u] = x > 1 ? __ldg(p.lnI + x) : 0.0;  // ln 1 = 0: singletons (most occupied slots) need no table read
          e[u] = x;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) tab[j0 + u * GT] = EMPTY_KEY;
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (e[u]) a2 = fma(u32_to_double(e[u]), lnx[u] - lbv[u], a2);
          N2 += e[u];
        }
      }
    }
    // ---- pass 3: folded 1D bins (two per word), four words = eight bins per thread in flight
    auto walk1d = [&](uint32_t* h1, int nw, const double* lb, double& acc, uint32_t& N) {
      constexpr int U = 4;
#pragma unroll 1
      for (int w0 = tg; w0 < nw; w0 += U * GT) {
        uint32_t v[U];
        double lbv[2 * U], lnx[2 * U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int w = w0 + u * GT;
          v[u] = w < nw ? h1[w] : 0u;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int w = w0 + u * GT;
          const uint32_t x0 = v[u] & 0xFFFF, x1 = v[u] >> 16;
          lbv[2 * u] = x0 ? __ldg(lb + 2 * w) : 0.0;
          lbv[2 * u + 1] = x1 ? __ldg(lb + 2 * w + 1) : 0.0;
          lnx[2 * u] = x0 > 1 ? __ldg(p.lnI + x0) : 0.0;
          lnx[2 * u + 1] = x1 > 1 ? __ldg(p.lnI + x1) : 0.0;
          if (v[u]) h1[w] = 0;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint32_t x0 = v[u] & 0xFFFF, x1 = v[u] >> 16;
          if (x0) acc = fma(u32_to_double(x0), lnx[2 * u] - lbv[2 * u], acc);
          if (x1) acc = fma(u32_to_double(x1), lnx[2 * u + 1] - lbv[2 * u + 1], acc);
          N += x0 + x1;
        }
      }
    };
    walk1d(h1a, nw1, lb1a, a1a, N1a);
    walk1d(h1b, nw2, lb1b, a1b, N1b);
    if (EXTRA && p.poisson) {  // no 1D statistics: their slots carry the Poisson sums through the reduction (pz_xq <= N2)
      a1a = pz_lg0; a1b = pz_lg1; N1a = pz_xq; N1b = 0;
    }
    // ---- reduce: warp level, then across the group's warps through shared memory
    // N2 | N1a << 10 | N1b << 20 : every total is <= WCAP < 1024
    uint32_t nn = __reduce_add_sync(0xffffffffu, N2 | (N1a << 10) | (N1b << 20));
    if (has_flags) count = __reduce_add_sync(0xffffffffu, count);
    if (snp_mode) nall = __reduce_add_sync(0xffffffffu, nall);
    a2 = warp_sum(a2); a1a = warp_sum(a1a); a1b = warp_sum(a1b);
    if (G > 1) {
      if (lane == 0) {
        double* rd = reinterpret_cast<double*>(red + wg * 10);
        rd[0] = a2; rd[1] = a1a; rd[2] = a1b;
        red[wg * 10 + 6] = nn; red[wg * 10 + 7] = (uint32_t)count; red[wg * 10 + 8] = (uint32_t)nall;
      }
      gsync();
      if (wg == 0) {
        a2 = a1a = a1b = 0.0; nn = 0; count = 0; nall = 0;
#pragma unroll
        for (int w = 0; w < G; ++w) {
          const double* rd = reinterpret_cast<const double*>(red + w * 10);
          a2 += rd[0]; a1a += rd[1]; a1b += rd[2];
          nn += red[w * 10 + 6]; count += (int)red[w * 10 + 7]; nall += (int)red[w * 10 + 8];
        }
      }
    }
    if (EXTRA && p.poisson) {
      // the whole group's sums (the host asks for one warp per window, but panels too wide for eight tables in 200 KB get
      // G = 2 or 4): lgamma(x + 1) in a1a, lgamma(x + 2) in a1b, the SNPs of the bins with q != 0 in N1a
      if (wg == 0 && lane == 0) {
        if (!has_flags) count = cnt;
        const int total = (int)(nn & 0x3FF);
        p.r_count[id] = count;
        p.r_flags[id] = 0;
        p.r_T2[id] = poisson_finish(p, total, (double)((nn >> 10) & 0x3FF), a2, a1a, a1b);
        p.r_n2[id] = total;
        p.r_T1a[id] = 0.0; p.r_T1b[id] = 0.0; p.r_n1a[id] = 0; p.r_n1b[id] = 0;
      }
    } else
    if (wg == 0) {  // lanes 0..2 finish one statistic each (ln N from the multiplicity table, ln B precomputed)
      if (!has_flags) count = cnt;
      const int Nq = lane == 0 ? (int)(nn & 0x3FF) : (lane == 1 ? (int)((nn >> 10) & 0x3FF) : (int)(nn >> 20));
      const double aq = lane == 0 ? a2 : (lane == 1 ? a1a : a1b);
      bool none = false;
      double Tq = 0.0;
      if (lane < 3) Tq = clr_value(p, Nq, aq, p.B + g * 6, lane, none);
      const uint32_t nb = __ballot_sync(0xffffffffu, none) & 7u;  // bit q = statistic q is None
      if (lane == 0) {
        uint8_t f = (uint8_t)nb;  // TDSFS_F_T2D_NONE = 1, _P1_NONE = 2, _P2_NONE = 4
        if (p.snp_mode && nall == 0) f |= TDSFS_F_SKIPPED;
        p.r_count[id] = count;
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
    gsync();
  }
}

// One CTA per large window; dense scratch histograms in global memory (L2 resident), cleared by re-walking the window.
// CTA `cta` of `ncta` (256 threads each, one scratch slab per CTA) takes every ncta-th entry of the large-window list.
constexpr int LARGE_THREADS = 256;
__device__ __forceinline__ void score_large_windows(const ScoreParams& p, int cta, int ncta) {
  __shared__ double red_d[3][LARGE_THREADS / 32];
  __shared__ int red_i[5][LARGE_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nl = *p.nlarge;
  const long long sstride = (long long)p.bins2d + p.n1 + 1 + p.n2 + 1;
  uint32_t* h2 = p.scratch + (long long)cta * sstride;
  uint32_t* h1a = h2 + p.bins2d;
  uint32_t* h1b = h1a + p.n1 + 1;
  const uint32_t last = p.poisson ? 0xFFFFFFFFu : (uint32_t)p.bins2d - 1;
  for (int w = cta; w < nl; w += ncta) {
    const long long id = p.large[w];
    const int lo = p.wlo[id], hi = p.whi[id];
    const int g = p.score_group ? p.score_group[p.wchrom[id]] : 0;
    const double* lb2 = p.lb2 + (long long)g * p.bins2d;
    const double* lb1a = p.lb1a + (long long)g * (p.n1 + 1);
    const double* lb1b = p.lb1b + (long long)g * (p.n2 + 1);
    int N2 = 0, N1a = 0, N1b = 0, nall = 0, count = 0;
    double a2 = 0.0, a1a = 0.0, a1b = 0.0;
    // Poisson score: sums of lgamma(x + 1) and lgamma(x + 2) over the populated bins with q != 0, and their SNPs (rows that
    // fail the spectrum filter or are monomorphic count in a window's rows but not in its total: total <= 1 happens here too)
    double pz_lg0 = 0.0, pz_lg1 = 0.0;
    int pz_xq = 0;
    for (int s = lo + tid; s < hi; s += LARGE_THREADS) {
      const uint2 r = load_rec(p.rec, p.fmt, s, p.n1, p.n2, p.C2);
      const uint32_t k = r.x, a = r.y;
      count += p.flags ? ((p.flags[s] >> 1) & 1) : 1;
      nall += k != 0;
      if (k != 0 && k != last) { atomicAdd(h2 + k, 1u); ++N2; }
      const int fa = (int)(a & 0xFFFF), fb = (int)(a >> 16);
      if (fa) { atomicAdd(h1a + fa, 1u); ++N1a; }
      if (fb) { atomicAdd(h1b + fb, 1u); ++N1b; }
    }
    __syncthreads();
    // second walk: the first thread to reach a bin takes its whole count x (atomicExch clears it) and adds x (ln x - ln b)
    for (int s = lo + tid; s < hi; s += LARGE_THREADS) {
      const uint2 r = load_rec(p.rec, p.fmt, s, p.n1, p.n2, p.C2);
      const uint32_t k = r.x, a = r.y;
      if (k != 0 && k != last) {
        const uint32_t x = atomicExch(h2 + k, 0u);
        if (x && p.poisson) {
          if (lb2[k] != -INFINITY) {
            a2 = fma((double)x, lb2[k], a2);
            pz_lg0 += lgamma((double)x + 1.0);
            pz_lg1 += lgamma((double)x + 2.0);
            pz_xq += (int)x;
          }
        } else if (x) a2 = fma((double)x, ln_mult(p, x) - lb2[k], a2);
      }
      const int fa = (int)(a & 0xFFFF), fb = (int)(a >> 16);
      if (fa) {
        const uint32_t x = atomicExch(h1a + fa, 0u);
        if (x) a1a = fma((double)x, ln_mult(p, x) - lb1a[fa], a1a);
      }
      if (fb) {
        const uint32_t x = atomicExch(h1b + fb, 0u);
        if (x) a1b = fma((double)x, ln_mult(p, x) - lb1b[fb], a1b);
      }
    }
    // block reduce
    if (p.poisson) { a1a = pz_lg0; a1b = pz_lg1; N1a = pz_xq; }  // reduced in the slots of the (unused) 1D statistics
    double dv[3] = {a2, a1a, a1b};
    int iv[5] = {N2, N1a, N1b, nall, count};
    for (int q = 0; q < 3; ++q) { dv[q] = warp_sum(dv[q]); if (lane == 0) red_d[q][warp] = dv[q]; }
    for (int q = 0; q < 5; ++q) { iv[q] = warp_sum(iv[q]); if (lane == 0) red_i[q][warp] = iv[q]; }
    __syncthreads();
    if (tid == 0) {
      for (int q = 0; q < 3; ++q) { double t = 0; for (int x = 0; x < LARGE_THREADS / 32; ++x) t += red_d[q][x]; dv[q] = t; }
      for (int q = 0; q < 5; ++q) { int t = 0; for (int x = 0; x < LARGE_THREADS / 32; ++x) t += red_i[q][x]; iv[q] = t; }
      if (p.poisson) {
        p.r_count[id] = iv[4];
        p.r_flags[id] = 0;
        p.r_T2[id] = poisson_finish(p, iv[0], (double)iv[1], dv[0], dv[1], dv[2]);
        p.r_n2[id] = iv[0];
        p.r_T1a[id] = 0.0; p.r_T1b[id] = 0.0; p.r_n1a[id] = 0; p.r_n1b[id] = 0;
      } else {
        write_result(p, id, iv[4], iv[3], iv[0], iv[1], iv[2], dv[0], dv[1], dv[2], p.B + g * 6);
      }
    }
    __syncthreads();
  }
}
__global__ void __launch_bounds__(LARGE_THREADS) k3_score_large(const __grid_constant__ ScoreParams p) {
  score_large_windows(p, blockIdx.x, gridDim.x);
}

// (ref1, alt1, ref2, alt2) of SNP s before the fix-ups, and the heterozygous calls het1, het2 (0 for the counts entry),
// from the source rows: the counts entry or the B32 genotype matrix with runtime word counts
__device__ __forceinline__ void source_counts(const KeyParams& p, long long s, int& ref1, int& alt1, int& ref2, int& alt2,
                                              int& het1, int& het2) {
  if (p.cnt) {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(p.cnt) + s);
    ref1 = v.x & 0xFFFF; alt1 = v.x >> 16; ref2 = v.y & 0xFFFF; alt2 = v.y >> 16;
    het1 = het2 = 0;
    return;
  }
  const int RW = p.W1 + p.W2;
  const uint32_t* row = p.G + ((s >> 5) * RW) * BLK + (s & 31);
  int T[2] = {0, 0}, M[2] = {0, 0};
  het1 = het2 = 0;  // scalars, not a third indexed array: a caller that ignores them compiles to the same code without them
  for (int w = 0; w < RW; w += 2) {  // (lo plane, hi plane) of 32 samples; W1 and W2 are even
    const uint32_t l = row[(long long)w * BLK], h = row[(long long)(w + 1) * BLK];
    T[w >= p.W1] += __popc(l) + __popc(h);
    M[w >= p.W1] += __popc(h & ~l);
    (w >= p.W1 ? het2 : het1) += __popc(l & ~h);
  }
  alt1 = T[0] - M[0]; alt2 = T[1] - M[1];
  ref1 = 2 * (p.ns1 - M[0]) - alt1; ref2 = 2 * (p.ns2 - M[1]) - alt2;
}

// dense spectra of one window (calculate_2d_sfs / calculate_1d_sfs on window_data): 2D bins from the stored records,
// raw (unfolded) 1D alt counts recomputed from the source rows (counts entry or B32 genotype matrix)
__global__ void k_window_hist(const __grid_constant__ KeyParams p, int lo, int hi, uint32_t* h2, uint32_t* h1a, uint32_t* h1b) {
  for (long long s = lo + blockIdx.x * blockDim.x + threadIdx.x; s < hi; s += gridDim.x * blockDim.x) {
    const uint32_t k = load_rec(p.rec, p.fmt, s, p.n1, p.n2, p.C2).x;
    if (k) atomicAdd(h2 + k, 1u);
    int ref1, alt1, ref2, alt2, het1, het2;
    source_counts(p, s, ref1, alt1, ref2, alt2, het1, het2);
    if (row_filters(p, s, ref1, alt1, ref2, alt2)) {
      if (alt1 > 0 && alt1 < p.R1) atomicAdd(h1a + alt1, 1u);
      if (alt2 > 0 && alt2 < p.R2) atomicAdd(h1b + alt2, 1u);
    }
  }
}

// ------------------------------------------------------------------------------------------------ explicit likelihood
// calculate_likelihood_1D/_2D on explicit interior vectors: T = 2 sum x (ln(x/N) - ln(b/B))
__global__ void __launch_bounds__(256) k_likelihood(const long long* x, const double* b, long long n, double B, double* out,
                                                    int* flag) {
  __shared__ double sd[8];
  __shared__ long long sn[8];
  long long N = 0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) N += x[i];
  for (int o = 16; o; o >>= 1) N += __shfl_xor_sync(0xffffffffu, N, o);
  if ((threadIdx.x & 31) == 0) sn[threadIdx.x >> 5] = N;
  __syncthreads();
  N = 0;
  for (int i = 0; i < 8; ++i) N += sn[i];
  if (N == 0 || !(B != 0.0)) {
    if (threadIdx.x == 0) { *out = NAN; *flag = 1; }
    return;
  }
  const double lnN = log((double)N), lnB = log(B);
  double acc = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) {
    const long long xi = x[i];
    if (xi > 0) {
      const double bi = b[i];
      const double lb = bi > 0.0 ? log(bi) : (bi == 0.0 ? -INFINITY : NAN);
      acc += (double)xi * ((log((double)xi) - lnN) - (lb - lnB));
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sd[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int i = 0; i < 8; ++i) t += sd[i];
    *out = 2.0 * t;
    *flag = 0;
  }
}

// legacy Poisson composite score (reference calculate_p :249-289): sum over bins with non-zero expectation of
// poisson.logpmf(x, mu) = x ln mu - mu - lgamma(x + 1)
__global__ void __launch_bounds__(256) k_poisson(const long long* x, const double* mu, long long n, double* out) {
  __shared__ double sd[8];
  double acc = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) {
    const double m = mu[i];
    if (m != 0.0) {
      const double xi = (double)x[i];
      acc += (xi == 0.0 ? 0.0 : xi * log(m)) - m - lgamma(xi + 1.0);
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sd[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int i = 0; i < 8; ++i) t += sd[i];
    *out = t;
  }
}

// ------------------------------------------------------------------------------------------------ synthetic panel
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
__device__ __forceinline__ double u01(uint64_t h) { return (double)(h >> 11) * (1.0 / 9007199254740992.0); }

// one thread per (row, word): one bit plane of 32 calls.  Ancestral frequency log-uniform on [1/(8n), 1-1/(8n)], per-population
// drift ~ normal approximation of Balding-Nichols with F = fst, calls Binomial(2, p), iid missing.
__global__ void __launch_bounds__(256) k_synth(uint32_t* G, long long S, long long snp0, int W1, int W2, int ns1, int ns2,
                                               uint64_t seed, uint32_t miss_thr16, double fst) {
  const int RW = W1 + W2;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // word index in the B32 layout
  const long long nblk = (S + BLK - 1) / BLK;
  if (idx >= nblk * RW * BLK) return;
  const long long bw = idx / BLK;  // block * RW + word
  const long long row = (bw / RW) * BLK + (idx & (BLK - 1));
  const int w = (int)(bw % RW);
  if (row >= S) { G[idx] = 0u; return; }
  const int pop = w >= W1;
  const int wi = pop ? w - W1 : w;
  const int ns = pop ? ns2 : ns1;
  const uint64_t snp = (uint64_t)(snp0 + row);
  const uint64_t hs = mix64(seed ^ (snp * 0x9E3779B97F4A7C15ULL));
  const double nn = 4.0 * (ns1 + ns2);  // 8 n with n = (ns1+ns2)/2
  const double lo = 1.0 / nn, hi = 1.0 - 1.0 / nn;
  const double pa = lo * exp(u01(hs) * log(hi / lo));
  // drift: sum of 4 uniforms ~ N(0, 1/3) scaled to unit variance
  const uint64_t hd = mix64(hs + 0x632BE59BD9B4E019ULL * (uint64_t)(pop + 1));
  const double z = ((double)(hd & 0xFFFF) + (double)((hd >> 16) & 0xFFFF) + (double)((hd >> 32) & 0xFFFF) +
                    (double)(hd >> 48)) * (1.0 / 65536.0) - 2.0;
  double pp = pa + z * 1.7320508 * sqrt(fst * pa * (1.0 - pa));
  pp = fmin(fmax(pp, 0.0), 1.0);
  const uint32_t thr = (uint32_t)(pp * 4294967296.0 > 4294967295.0 ? 4294967295.0 : pp * 4294967296.0);
  uint32_t word = 0;
  const int plane = wi & 1;  // 0: lo bits of the codes, 1: hi bits
  for (int i = 0; i < 32; ++i) {
    const int sample = (wi >> 1) * 32 + i;
    if (sample >= ns) break;
    const uint64_t h1 = mix64(hs ^ ((uint64_t)(pop * 1000003 + sample + 1) * 0xD6E8FEB86659FD93ULL));
    const uint64_t h2 = mix64(h1);
    const uint32_t a1 = (uint32_t)h1 < thr, a2 = (uint32_t)(h1 >> 32) < thr;
    uint32_t code = (a1 + a2 == 0) ? 0u : (a1 + a2 == 1 ? 1u : 3u);
    if ((uint32_t)(h2 & 0xFFFF) < miss_thr16) code = 2u;
    word |= ((code >> plane) & 1u) << i;
  }
  G[idx] = word;
}

}  // namespace tdsfs
