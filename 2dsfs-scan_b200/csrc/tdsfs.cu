// tdsfs.cu -- C ABI of libtdsfs.so (see include/tdsfs.h) over the kernels in tdsfs_kernels.cuh.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC (see build.py)
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <cub/device/device_scan.cuh>
#include <nvtx3/nvToolsExt.h>

#include "tdsfs_kernels.cuh"
#include "tdsfs_fused.cuh"
#include "tdsfs_diversity.cuh"
#include "tdsfs_ld.cuh"

using namespace tdsfs;

#define TDSFS_VERSION 204

static thread_local std::string g_err;

// NVTX range around every phase of the pass (count kernel, window boundaries, exchange, finalize, finish): visible to
// Nsight Systems / Compute timelines, free when no tool is attached
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

static int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

// a rank that never arrives flags an error instead of hanging the others: ~60 s of SM cycles by default (ranks of a real job may
// reach the exchange seconds apart), TDSFS_PEER_TIMEOUT_S overrides
static long long peer_timeout_cycles() {
  static long long v = 0;
  if (!v) {
    double s = 60.0;
    if (const char* e = getenv("TDSFS_PEER_TIMEOUT_S")) s = std::max(0.001, atof(e));
    v = (long long)(s * 2.0e9);
  }
  return v;
}
#define PEER_TIMEOUT_CYCLES peer_timeout_cycles()

#define CK(call)                                                                                        \
  do {                                                                                                  \
    cudaError_t e__ = (call);                                                                           \
    if (e__ != cudaSuccess) return fail(TDSFS_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                                        __FILE__, __LINE__);                                            \
  } while (0)
#define CKR(call)              \
  do {                         \
    int r__ = (call);          \
    if (r__) return r__;       \
  } while (0)

enum { EV_BG0, EV_K1, EV_FIN0, EV_FIN1, EV_SC0, EV_K2, EV_K3S, EV_K3L, EV_X0, EV_X1, NEV };

struct Chunk {
  long long r0, r1;
  cudaEvent_t ev;
};

// Candidate-window offsets per chromosome of one (size, mode), on the host and the device (cached_candidates): computed
// and uploaded again only when (size, mode) changes, so that a steady-state call needs no host round trip.
struct CandCache {
  long long W = -1;                   // (size, mode) the offsets are of; -1: none
  int snp = -1;
  std::vector<long long> off;         // [C + 1]
  long long* d_off = nullptr;
  bool holds(long long size, bool snp_mode) const { return W == size && snp == (int)snp_mode; }
};

// Workspace and results of one per-window pass over the candidate windows of (size, mode) (tdsfs_diversity_*,
// tdsfs_neutrality_*, tdsfs_wcfst_*): its candidate offsets, window boundaries, segment list, scan scratch, per-segment sums, per-window
// results and events.
struct WindowPass {
  WindowPass(const char* name, size_t part_bytes, int n_i32, int n_f64)
      : name(name), part_bytes(part_bytes), n_i32(n_i32), n_f64(n_f64) {}
  const char* name;                   // NVTX range of a call
  size_t part_bytes;                  // size of the pass's per-segment sums (DivPart, NeutPart, WcPart)
  int n_i32, n_f64;                   // result columns of the pass in d_i32 / d_f64
  CandCache cand;
  long long cap = 0, ncand = 0;       // windows the per-window arrays hold / of the last call
  size_t tmp_bytes = 0;
  int32_t *d_wlo = nullptr, *d_whi = nullptr, *d_wchrom = nullptr, *d_count = nullptr;
  int32_t* d_large = nullptr;         // never written: a per-window pass has no "large window" split
  int* d_nlarge = nullptr;
  long long *d_wstart = nullptr, *d_wend = nullptr, *d_nseg = nullptr, *d_segoff = nullptr;
  uint8_t* d_flags = nullptr;
  void* d_tmp = nullptr;              // CUB scan scratch
  int32_t* d_i32[4] = {};             // [cap] the pass's int32 and fp64 result columns, each in the order of its result
  double* d_f64[6] = {};              // struct in include/tdsfs.h
  void* d_part = nullptr;             // [part_cap] per-segment sums
  long long part_cap = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // around the segment and finish kernels (tdsfs_timings)
  bool ready = false, timed = false;  // results of the last call are on the device / its events were recorded
  SegList segs() const { return SegList{d_wlo, d_whi, ncand, d_segoff}; }
};

struct tdsfs_ctx {
  int device = 0, sm_count = 148;
  cudaStream_t stream = nullptr, own_stream = nullptr, copy_stream = nullptr;
  bool sync = true;
  // panel
  int n1 = 0, n2 = 0, fold = 1, R1 = 0, R2 = 0, bins2d = 0;
  // data
  long long S = 0;
  int C = 0;
  const uint32_t* dG = nullptr;
  bool own_G = false;
  // pooled device buffers reused across loads (sizes in bytes)
  void *pool_G = nullptr, *pool_cnt = nullptr, *pool_pos = nullptr, *pool_flags = nullptr, *pool_off = nullptr, *pool_tmp = nullptr;
  size_t cap_G = 0, cap_cnt = 0, cap_pos = 0, cap_flags = 0, cap_off = 0, cap_tmp = 0;
  int W1 = 0, W2 = 0, ns1 = 0, ns2 = 0;
  const uint16_t* dCnt = nullptr;
  bool own_cnt = false;
  const int32_t* dPos = nullptr;
  bool own_pos = false;
  bool loaded = false;     // a (possibly empty) data set is loaded
  bool genotypes = false;  // ... through tdsfs_load_genotypes: the 2-bit calls are on the device
  const uint8_t* dFlags = nullptr;
  bool own_flags = false;
  tdsfs_fixup_t* dFix = nullptr;
  long long nfix = 0;
  std::vector<long long> h_off;
  std::vector<long long> h_last;  // last position per chromosome (-1 = empty)
  long long* d_off = nullptr;
  std::vector<Chunk> chunks;
  // keys
  void* d_rec = nullptr;   // per-SNP records (RecFmt: 4-byte narrow or 8-byte wide)
  long long key_cap = 0;
  bool keys_ready = false;
  RecFmt fmt = {0, 0, 0, 0};  // format of the records d_rec currently holds
  bool force_wide = false;    // a SNP did not fit the narrow record: wide records until the next load
  // fused scan: window sums written by k1_fused for the plan (fused_W, fused_snp)
  double* d_ws = nullptr;
  long long ws_cap = 0;
  long long fused_W = -1;
  int fused_snp = -1;
  bool ws_ready = false;
  bool last_fused = false;    // the last scan was finished by k3_finish
  double* d_dxI = nullptr;
  // background
  int bg_mode = -1, NG = 0;
  long long gstride = 0;
  uint32_t* d_hist = nullptr;
  long long hist_words = 0;
  int32_t* d_bg_group = nullptr;
  int32_t* d_score_group = nullptr;
  bool per_chrom_scoring = false;
  double *d_lb2 = nullptr, *d_lb1a = nullptr, *d_lb1b = nullptr, *d_B = nullptr, *d_lnI = nullptr;
  unsigned long long* d_Bsum = nullptr;
  int table_groups = 0;
  bool float_bg = false, tables_ready = false, fin_timed = false;
  bool poisson_bg = false;            // the tables hold ln q of a normalised background (tdsfs_set_poisson_background)
  double pq_n = 0, pq_sum = 0, pq_lnsum = 0;
  bool tables_from_exchange = false;  // the merged exchange kernel (or the count kernel's tail) already built the tables of this background
  unsigned int* d_gridbar = nullptr;  // grid barrier of the count kernel's tail: arrivals, phase
  unsigned long long* d_stamps = nullptr;  // diagnostics (TDSFS_TAIL_STAMPS=1): clock64 of CTA 0 at the phases of the tail
  bool want_tail_exchange = false;    // tdsfs_step_bp: the next tdsfs_background also exchanges the histogram (peer memory) in its tail
  bool x_timed = false;
  int score_group_warps = 1;  // warps per window in the shared-memory scorer (1, 2 or 4)
  int* d_err = nullptr;
  // peer-memory exchange of the background histogram (tdsfs_peer_*)
  int peer_rank = -1, peer_world = 0;
  uint32_t* peer_hist[PEER_MAX] = {};
  unsigned long long* peer_flags[PEER_MAX] = {};
  unsigned long long* d_peer_flags = nullptr;  // this rank's flag array
  uint32_t* peer_exported_hist = nullptr;
  long long peer_words = 0;
  bool peer_ready = false;
  // windows / results
  long long ncand = 0, cand_cap = 0;
  CandCache cand;
  int groups_mode = -1, groups_chrom = -1;  // what d_bg_group / d_score_group currently hold
  // window plan launched ahead of the scan on a side stream (tdsfs_plan_bp / _snp)
  cudaStream_t plan_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_plan = nullptr, ev_plan0 = nullptr;
  long long plan_W = -1;
  int plan_snp = -1;
  bool planned_last = false;
  int32_t *d_wlo = nullptr, *d_whi = nullptr, *d_wchrom = nullptr, *d_large = nullptr;
  long long *d_wstart = nullptr, *d_wend = nullptr;
  int* d_nlarge = nullptr;
  int32_t *r_count = nullptr, *r_n2 = nullptr, *r_n1a = nullptr, *r_n1b = nullptr;
  double *r_T2 = nullptr, *r_T1a = nullptr, *r_T1b = nullptr;
  uint8_t* r_flags = nullptr;
  uint32_t* d_scratch = nullptr;
  int large_ctas = 0;
  unsigned long long* d_work = nullptr;  // window hand-out counter of the scorer (monotonic, never reset)
  unsigned long long work_base = 0;
  bool results_ready = false;
  // whole asynchronous pass captured as a CUDA graph (tdsfs_step_bp): replayed while nothing it depends on changes
  unsigned long long generation = 0;  // bumped by every load / panel / stream / peer change
  cudaGraphExec_t step_exec = nullptr;
  unsigned long long step_gen = 0, warm_gen = 0;
  long long step_W = -1, warm_W = -1;
  int step_mode = -1, warm_mode = -1;
  long long step_launches = 0;
  bool step_graphs_off = false;       // capture failed once: run eagerly from then on
  // per-window passes over the scan's candidate windows: each has its own workspace and results, so that it never touches
  // the scan's plan, window buffers or unfetched results, nor the other pass's
  WindowPass div{"tdsfs:diversity (FST, pi, dxy)", sizeof(DivPart), 1, 4};                 // tdsfs_diversity_*
  WindowPass neut{"tdsfs:neutrality (theta_W, Tajima's D)", sizeof(NeutPart), 4, 6};      // tdsfs_neutrality_*
  WindowPass wc{"tdsfs:Weir and Cockerham FST", sizeof(WcPart), 1, 4};                    // tdsfs_wcfst_*
  double* d_neut_tab = nullptr;       // a1(n) for n in [0, neut_tab_n], then a2(n) for the same n
  long long neut_tab_n = -1;
  long long n_allele_max = 0;         // the largest n_i = ref_i + alt_i a row of the loaded data can reach
  // LD pruning (tdsfs_ld_prune): a workspace of its own, so that a pending plan, the scan's results, the step graph and the
  // window passes' results survive it
  uint32_t* d_ld_mask = nullptr;      // [S * mask words] pair bits of k_ld_pairs
  long long ld_mask_cap = 0;
  uint8_t* d_ld_keep = nullptr;       // [S]
  long long ld_keep_cap = 0;
  unsigned long long* d_ld_n = nullptr;  // kept rows
  cudaEvent_t ev_ld[3] = {};          // before k_ld_pairs, between the kernels, after k_ld_resolve (tdsfs_timings)
  bool ld_timed = false;
  // instrumentation
  cudaEvent_t ev[NEV] = {};
  float ms[14] = {};
  long long launches = 0;
};

static void peer_unmap(tdsfs_ctx* c);

template <typename T>
static int dev_alloc(T** p, long long n) {
  CK(cudaMalloc((void**)p, (size_t)std::max<long long>(n, 1) * sizeof(T)));
  return 0;
}
template <typename T>
static void dev_free(T*& p) {
  if (p) cudaFree((void*)p);
  p = nullptr;
}

static bool is_device_ptr(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// device-side error word -> return code (bit0 range, bit2 peer timeout, bit3 narrow-record overflow)
static int deferred_error(tdsfs_ctx* c, int err) {
  if (err & 4) return fail(TDSFS_ERR_CUDA, "peer exchange: a rank did not reach the barrier in time; the background is incomplete");
  if (err & 16) return fail(TDSFS_ERR_CUDA, "count kernel: its CTAs did not all reach the grid barrier in time; the background tables are incomplete");
  if (err & 1) return fail(TDSFS_ERR_RANGE, "an allele count exceeds 2n of the declared panel (n1=%d, n2=%d)", c->n1, c->n2);
  if (err & 8) {
    c->force_wide = true;
    c->ws_ready = false;
    return fail(TDSFS_ERR_RETRY, "a SNP's missing-call counts do not fit the 4-byte record; the handle now uses 8-byte records: run the pass again");
  }
  return 0;
}

static int finish(tdsfs_ctx* c) {
  if (c->sync) CK(cudaStreamSynchronize(c->stream));
  return 0;
}

// ------------------------------------------------------------------------------------------------ lifetime
extern "C" const char* tdsfs_last_error(void) { return g_err.c_str(); }
extern "C" int tdsfs_version(void) { return TDSFS_VERSION; }

extern "C" int tdsfs_create(int device, tdsfs_t** out) {
  if (!out) return fail(TDSFS_ERR_ARG, "out is NULL");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(TDSFS_ERR_CUDA, "no CUDA device available: libtdsfs has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(TDSFS_ERR_ARG, "device %d out of range (%d devices)", device, ndev);
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(TDSFS_ERR_CUDA, "device %s is sm_%d%d; libtdsfs is built for sm_100a only", prop.name, prop.major, prop.minor);
  tdsfs_ctx* c = new tdsfs_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  CK(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&c->plan_stream, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  CK(cudaEventCreate(&c->ev_plan));
  CK(cudaEventCreate(&c->ev_plan0));
  c->stream = c->own_stream;
  for (int i = 0; i < NEV; ++i) CK(cudaEventCreate(&c->ev[i]));
  for (WindowPass* w : {&c->div, &c->neut, &c->wc}) {
    CK(cudaEventCreate(&w->ev0));
    CK(cudaEventCreate(&w->ev1));
  }
  for (cudaEvent_t& e : c->ev_ld) CK(cudaEventCreate(&e));
  CKR(dev_alloc(&c->d_ld_n, 1));
  CKR(dev_alloc(&c->d_err, 1));
  CKR(dev_alloc(&c->d_nlarge, 1));
  CKR(dev_alloc(&c->d_lnI, LN_TABLE));
  CK(cudaMemsetAsync(c->d_err, 0, sizeof(int), c->stream));
  k_ln_int_table<<<(LN_TABLE + 255) / 256, 256, 0, c->stream>>>(c->d_lnI, LN_TABLE);
  c->launches++;
  CK(cudaGetLastError());
  CKR(dev_alloc(&c->d_gridbar, 2));
  CK(cudaMemsetAsync(c->d_gridbar, 0, 2 * sizeof(unsigned int), c->stream));
  if (getenv("TDSFS_TAIL_STAMPS")) {
    CKR(dev_alloc(&c->d_stamps, 8));
    CK(cudaMemsetAsync(c->d_stamps, 0, 8 * sizeof(unsigned long long), c->stream));
  }
  CKR(dev_alloc(&c->d_dxI, LN_TABLE));
  k_dx_table<<<(LN_TABLE + 255) / 256, 256, 0, c->stream>>>(c->d_dxI, LN_TABLE);
  c->launches++;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(c->stream));
  *out = c;
  return 0;
}

static int pool_get(void** pool, size_t* cap, size_t bytes, void** out) {
  if (bytes > *cap) {
    if (*pool) cudaFree(*pool);
    *pool = nullptr;
    *cap = 0;
    CK(cudaMalloc(pool, std::max<size_t>(bytes, 256)));
    *cap = std::max<size_t>(bytes, 256);
  }
  *out = *pool;
  return 0;
}

static void drop_step_graph(tdsfs_ctx* c) {
  if (c->step_exec) cudaGraphExecDestroy(c->step_exec);
  c->step_exec = nullptr;
  c->generation++;
}

static void free_data(tdsfs_ctx* c) {
  drop_step_graph(c);
  // a window plan that no scan consumed may still be reading the (pooled) position / offset arrays on the side stream
  if (c->plan_W >= 0 && c->ev_plan) cudaStreamWaitEvent(c->stream, c->ev_plan, 0);
  c->dG = nullptr; c->dCnt = nullptr; c->dPos = nullptr; c->dFlags = nullptr;
  c->own_G = c->own_cnt = c->own_pos = c->own_flags = false;
  c->loaded = c->genotypes = false;
  dev_free(c->dFix);
  c->nfix = 0;
  c->d_off = nullptr;  // pooled (pool_off)
  for (auto& ch : c->chunks) if (ch.ev) cudaEventDestroy(ch.ev);
  c->chunks.clear();
  c->keys_ready = c->tables_ready = c->results_ready = false;
  c->cand.W = -1;
  c->groups_mode = -1;
  c->plan_W = -1;
  c->ws_ready = false;
  c->force_wide = false;
  for (WindowPass* w : {&c->div, &c->neut, &c->wc}) {
    w->cand.W = -1;
    w->ready = false;
  }
  c->n_allele_max = 0;
}

// the per-window arrays of pass w
static void free_pass_windows(WindowPass& w) {
  dev_free(w.d_wlo); dev_free(w.d_whi); dev_free(w.d_wchrom); dev_free(w.d_count); dev_free(w.d_wstart); dev_free(w.d_wend);
  dev_free(w.d_nseg); dev_free(w.d_segoff); dev_free(w.d_flags); dev_free(w.d_tmp);
  for (int32_t*& a : w.d_i32) dev_free(a);
  for (double*& a : w.d_f64) dev_free(a);
}

static void free_window_pass(WindowPass& w) {
  free_pass_windows(w);
  dev_free(w.cand.d_off); dev_free(w.d_large); dev_free(w.d_nlarge); dev_free(w.d_part);
  if (w.ev0) cudaEventDestroy(w.ev0);
  if (w.ev1) cudaEventDestroy(w.ev1);
}

extern "C" void tdsfs_destroy(tdsfs_t* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  drop_step_graph(c);
  free_data(c);
  if (c->pool_G) cudaFree(c->pool_G);
  if (c->pool_cnt) cudaFree(c->pool_cnt);
  if (c->pool_pos) cudaFree(c->pool_pos);
  if (c->pool_flags) cudaFree(c->pool_flags);
  if (c->pool_off) cudaFree(c->pool_off);
  if (c->pool_tmp) cudaFree(c->pool_tmp);
  peer_unmap(c);
  dev_free(c->d_peer_flags);
  dev_free(c->d_work);
  if (c->d_rec) cudaFree(c->d_rec);
  dev_free(c->d_hist); dev_free(c->d_bg_group); dev_free(c->d_score_group);
  dev_free(c->d_lb2); dev_free(c->d_lb1a); dev_free(c->d_lb1b); dev_free(c->d_B); dev_free(c->d_Bsum); dev_free(c->d_lnI);
  dev_free(c->d_err); dev_free(c->cand.d_off); dev_free(c->d_wlo); dev_free(c->d_whi); dev_free(c->d_wchrom);
  dev_free(c->d_large); dev_free(c->d_wstart); dev_free(c->d_wend); dev_free(c->d_nlarge);
  dev_free(c->r_count); dev_free(c->r_n2); dev_free(c->r_n1a); dev_free(c->r_n1b); dev_free(c->r_T2); dev_free(c->r_T1a);
  dev_free(c->r_T1b); dev_free(c->r_flags); dev_free(c->d_scratch);
  for (int i = 0; i < NEV; ++i) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
  dev_free(c->d_dxI); dev_free(c->d_ws); dev_free(c->d_gridbar); dev_free(c->d_stamps);
  free_window_pass(c->div);
  free_window_pass(c->neut);
  free_window_pass(c->wc);
  dev_free(c->d_neut_tab);
  dev_free(c->d_ld_mask); dev_free(c->d_ld_keep); dev_free(c->d_ld_n);
  for (cudaEvent_t e : c->ev_ld) if (e) cudaEventDestroy(e);
  cudaStreamDestroy(c->own_stream);
  cudaStreamDestroy(c->copy_stream);
  cudaStreamDestroy(c->plan_stream);
  cudaEventDestroy(c->ev_fork); cudaEventDestroy(c->ev_plan); cudaEventDestroy(c->ev_plan0);
  delete c;
}

extern "C" int tdsfs_set_stream(tdsfs_t* c, void* s) {
  if (!c) return fail(TDSFS_ERR_ARG, "ctx is NULL");
  c->stream = s ? (cudaStream_t)s : c->own_stream;
  drop_step_graph(c);
  return 0;
}

extern "C" int tdsfs_set_sync(tdsfs_t* c, int sync) {
  if (!c) return fail(TDSFS_ERR_ARG, "ctx is NULL");
  c->sync = sync != 0;
  return 0;
}

extern "C" int tdsfs_set_panel(tdsfs_t* c, int32_t n1, int32_t n2, int32_t fold) {
  if (!c) return fail(TDSFS_ERR_ARG, "ctx is NULL");
  if (n1 < 1 || n2 < 1 || n1 > 32767 || n2 > 32767) return fail(TDSFS_ERR_ARG, "panel sizes must be in [1, 32767] (got %d, %d)", n1, n2);
  long long bins = (long long)(2 * n1 + 1) * (2 * n2 + 1);
  if (bins > 0x7FFFFFFFLL) return fail(TDSFS_ERR_ARG, "2D spectrum too large: (2 n1 + 1)(2 n2 + 1) = %lld bins exceeds 2^31 - 1", bins);
  CK(cudaSetDevice(c->device));
  drop_step_graph(c);
  c->n1 = n1; c->n2 = n2; c->fold = fold != 0;
  c->R1 = 2 * n1 + 1; c->R2 = 2 * n2 + 1; c->bins2d = (int)bins;
  c->keys_ready = c->tables_ready = c->results_ready = false;
  c->bg_mode = -1;
  // everything sized by the spectrum shape is rebuilt for the new panel
  dev_free(c->d_lb2); dev_free(c->d_lb1a); dev_free(c->d_lb1b); dev_free(c->d_B); dev_free(c->d_Bsum);
  c->table_groups = 0;
  dev_free(c->d_scratch);
  peer_unmap(c);  // peers must have closed their mappings of this histogram (tdsfs_peer_close) before it is freed
  c->peer_exported_hist = nullptr;
  dev_free(c->d_hist);
  c->hist_words = 0;
  return 0;
}

// ------------------------------------------------------------------------------------------------ data
template <typename T>
static int adopt_or_upload(tdsfs_ctx* c, const T* src, long long n, const T** dst, bool* own, void** pool, size_t* cap) {
  if (is_device_ptr(src)) {
    *dst = src;
    *own = false;
    return 0;
  }
  void* d = nullptr;
  CKR(pool_get(pool, cap, (size_t)n * sizeof(T), &d));
  CK(cudaMemcpyAsync(d, src, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  *dst = (const T*)d;
  *own = true;
  return 0;
}

static int load_common(tdsfs_ctx* c, long long S, const int32_t* pos, const long long* chrom_off, int C, const uint8_t* flags,
                       bool need_flag_copy) {
  if (S < 0 || S > 0x7FFFFF00LL) return fail(TDSFS_ERR_ARG, "S = %lld out of range", S);
  if (C < 0 || !chrom_off || (!pos && S > 0)) return fail(TDSFS_ERR_ARG, "pos / chrom_off missing or C < 0");
  if (C == 0 && S != 0) return fail(TDSFS_ERR_ARG, "no chromosomes but S = %lld", S);
  if (chrom_off[0] != 0 || chrom_off[C] != S) return fail(TDSFS_ERR_ARG, "chrom_off must start at 0 and end at S");
  for (int i = 0; i < C; ++i)
    if (chrom_off[i + 1] < chrom_off[i]) return fail(TDSFS_ERR_ARG, "chrom_off not monotone");
  c->S = S;
  c->C = C;
  c->h_off.assign(chrom_off, chrom_off + C + 1);
  {
    void* d = nullptr;  // pooled: no cudaMalloc per load (the per-replicate sims path loads thousands of small panels)
    CKR(pool_get(&c->pool_off, &c->cap_off, (size_t)(C + 1) * sizeof(long long), &d));
    c->d_off = (long long*)d;
  }
  CK(cudaMemcpyAsync(c->d_off, chrom_off, (size_t)(C + 1) * sizeof(long long), cudaMemcpyHostToDevice, c->stream));
  if (S > 0) CKR(adopt_or_upload(c, pos, S, &c->dPos, &c->own_pos, &c->pool_pos, &c->cap_pos));
  else {  // an empty shard (a rank of a sharded scan with no rows): a valid, empty position array
    void* d = nullptr;
    CKR(pool_get(&c->pool_pos, &c->cap_pos, 256, &d));
    c->dPos = (const int32_t*)d;
    c->own_pos = true;
  }
  if (flags && S > 0) {
    if (need_flag_copy && is_device_ptr(flags)) {
      void* d = nullptr;
      CKR(pool_get(&c->pool_flags, &c->cap_flags, (size_t)S, &d));
      CK(cudaMemcpyAsync(d, flags, (size_t)S, cudaMemcpyDeviceToDevice, c->stream));
      c->dFlags = (const uint8_t*)d;
      c->own_flags = true;
    } else {
      CKR(adopt_or_upload(c, flags, S, &c->dFlags, &c->own_flags, &c->pool_flags, &c->cap_flags));
    }
  }
  // last position of every chromosome (sizes the fixed-bp candidate list)
  c->h_last.assign(C, -1);
  if (!is_device_ptr(pos)) {
    for (int i = 0; i < C; ++i)
      if (chrom_off[i + 1] > chrom_off[i]) c->h_last[i] = pos[chrom_off[i + 1] - 1];
  } else {
    for (int i = 0; i < C; ++i)
      if (chrom_off[i + 1] > chrom_off[i]) {
        int32_t v;
        CK(cudaMemcpyAsync(&v, pos + chrom_off[i + 1] - 1, sizeof v, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        c->h_last[i] = v;
      }
  }
  if (S > c->key_cap) {
    if (c->d_rec) cudaFree(c->d_rec);
    c->d_rec = nullptr;
    CK(cudaMalloc(&c->d_rec, (size_t)std::max<long long>(S, 1) * sizeof(uint2)));  // sized for the wide form
    c->key_cap = S;
  }
  return 0;
}

extern "C" int tdsfs_load_counts(tdsfs_t* c, const uint16_t* cnt, int64_t S, const int32_t* pos, const int64_t* chrom_off,
                                 int32_t C, const uint8_t* snp_flags) {
  if (!c || (!cnt && S > 0)) return fail(TDSFS_ERR_ARG, "ctx / cnt is NULL");
  if (!c->bins2d) return fail(TDSFS_ERR_STATE, "tdsfs_set_panel first");
  CK(cudaSetDevice(c->device));
  free_data(c);
  CKR(load_common(c, S, pos, (const long long*)chrom_off, C, snp_flags, false));
  if (S > 0) {
    CKR(adopt_or_upload(c, cnt, S * 4, &c->dCnt, &c->own_cnt, &c->pool_cnt, &c->cap_cnt));
    if (((uintptr_t)c->dCnt & 7) != 0) return fail(TDSFS_ERR_ARG, "cnt must be 8-byte aligned");
  }
  c->n_allele_max = 2 * 65535;
  c->loaded = true;
  return finish(c);
}

extern "C" int tdsfs_load_genotypes(tdsfs_t* c, const void* G, int64_t S, int32_t words1, int32_t words2, int32_t ns1,
                                    int32_t ns2, const int32_t* pos, const int64_t* chrom_off, int32_t C,
                                    const tdsfs_fixup_t* fixups, int64_t n_fixups, const uint8_t* snp_flags) {
  if (!c || (!G && S > 0)) return fail(TDSFS_ERR_ARG, "ctx / G is NULL");
  if (!c->bins2d) return fail(TDSFS_ERR_STATE, "tdsfs_set_panel first");
  if (words1 < 2 || words2 < 2 || (words1 & 1) || (words2 & 1) || ns1 < 0 || ns2 < 0 || ns1 > words1 * 16 || ns2 > words2 * 16)
    return fail(TDSFS_ERR_ARG, "bad genotype geometry (words %d/%d, samples %d/%d): a population is an even number of words, 32 samples per (lo, hi) pair",
                words1, words2, ns1, ns2);
  if (ns1 > 65535 / 2 || ns2 > 65535 / 2) return fail(TDSFS_ERR_ARG, "more than 32767 samples per population");
  CK(cudaSetDevice(c->device));
  free_data(c);
  const bool has_fix = fixups && n_fixups > 0;
  CKR(load_common(c, S, pos, (const long long*)chrom_off, C, snp_flags, has_fix));
  c->W1 = words1; c->W2 = words2; c->ns1 = ns1; c->ns2 = ns2;
  c->genotypes = true;
  c->n_allele_max = 2LL * std::max(ns1, ns2);
  const long long RW = words1 + words2;
  if (has_fix) {
    // flag bit2 marks rows that own fix-ups; build (or extend) the flag array on the host side
    std::vector<tdsfs_fixup_t> hf(fixups, fixups + n_fixups);
    if (!std::is_sorted(hf.begin(), hf.end(), [](const tdsfs_fixup_t& a, const tdsfs_fixup_t& b) { return a.snp < b.snp; }))
      return fail(TDSFS_ERR_ARG, "fixups must be sorted by snp");
    std::vector<uint8_t> hflags((size_t)S, 3);
    if (c->dFlags) {
      CK(cudaMemcpyAsync(hflags.data(), c->dFlags, (size_t)S, cudaMemcpyDeviceToHost, c->stream));
      CK(cudaStreamSynchronize(c->stream));
      for (auto& f : hflags) f &= 3;
    }
    for (auto& f : hf) {
      if (f.snp < 0 || f.snp >= S || (f.pop != 0 && f.pop != 1)) return fail(TDSFS_ERR_ARG, "fixup out of range");
      hflags[(size_t)f.snp] |= 4;
    }
    for (size_t i = 0, j; i < hf.size(); i = j) {  // the fix-ups of one (row, population) add up
      long long dn[2] = {0, 0};
      for (j = i; j < hf.size() && hf[j].snp == hf[i].snp; ++j) dn[hf[j].pop] += (long long)hf[j].dref + hf[j].dalt;
      c->n_allele_max = std::max(c->n_allele_max, 2LL * std::max(ns1, ns2) + std::max(dn[0], dn[1]));
    }
    if (!c->own_flags) {
      void* d = nullptr;
      CKR(pool_get(&c->pool_flags, &c->cap_flags, (size_t)S, &d));
      c->dFlags = (const uint8_t*)d;
      c->own_flags = true;
    }
    CK(cudaMemcpyAsync((void*)c->dFlags, hflags.data(), (size_t)S, cudaMemcpyHostToDevice, c->stream));
    CKR(dev_alloc(&c->dFix, n_fixups));
    CK(cudaMemcpyAsync(c->dFix, hf.data(), (size_t)n_fixups * sizeof(tdsfs_fixup_t), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->nfix = n_fixups;
  }
  c->loaded = true;
  if (S == 0) {
    c->chunks.push_back({0, 0, nullptr});
    return finish(c);
  }
  if (is_device_ptr(G)) {
    if (((uintptr_t)G & 15) != 0) return fail(TDSFS_ERR_ARG, "device G must be 16-byte aligned");
    c->dG = (const uint32_t*)G;
    c->own_G = false;
    c->chunks.push_back({0, S, nullptr});
  } else {
    // chunked asynchronous upload on the copy stream; tdsfs_background's count kernel consumes chunk by chunk
    void* dv = nullptr;
    const long long nblk = (S + BLK - 1) / BLK;
    const long long blk_bytes = RW * BLK * 4;
    CKR(pool_get(&c->pool_G, &c->cap_G, (size_t)(nblk * blk_bytes), &dv));
    uint32_t* d = (uint32_t*)dv;
    c->dG = d;
    c->own_G = true;
    long long chunk_bytes = 64LL << 20;
    if (const char* e = getenv("TDSFS_UPLOAD_CHUNK_KB")) chunk_bytes = std::max(1, atoi(e)) * 1024LL;  // test knob: many small chunks
    const long long blks_per_chunk = std::max<long long>(K1_ROWS / BLK, chunk_bytes / blk_bytes / (K1_ROWS / BLK) * (K1_ROWS / BLK));
    CK(cudaStreamSynchronize(c->stream));
    for (long long bb0 = 0; bb0 < nblk; bb0 += blks_per_chunk) {
      const long long bb1 = std::min<long long>(nblk, bb0 + blks_per_chunk);
      Chunk ch{bb0 * BLK, std::min<long long>(S, bb1 * BLK), nullptr};
      CK(cudaEventCreateWithFlags(&ch.ev, cudaEventDisableTiming));
      CK(cudaMemcpyAsync((uint8_t*)d + bb0 * blk_bytes, (const uint8_t*)G + bb0 * blk_bytes, (size_t)((bb1 - bb0) * blk_bytes),
                         cudaMemcpyHostToDevice, c->copy_stream));
      CK(cudaEventRecord(ch.ev, c->copy_stream));
      c->chunks.push_back(ch);
    }
    if (S == 0) c->chunks.push_back({0, 0, nullptr});
  }
  return finish(c);
}

// ------------------------------------------------------------------------------------------------ background
static int ensure_tables(tdsfs_ctx* c, int NG) {
  if (NG <= c->table_groups) return 0;
  dev_free(c->d_lb2); dev_free(c->d_lb1a); dev_free(c->d_lb1b); dev_free(c->d_B); dev_free(c->d_Bsum);
  CKR(dev_alloc(&c->d_lb2, (long long)NG * c->bins2d));
  CKR(dev_alloc(&c->d_lb1a, (long long)NG * (c->n1 + 1)));
  CKR(dev_alloc(&c->d_lb1b, (long long)NG * (c->n2 + 1)));
  CKR(dev_alloc(&c->d_B, (long long)NG * 6));
  CKR(dev_alloc(&c->d_Bsum, (long long)NG * 3 + 1));  // + the finalize kernel's CTA counter; the kernel leaves all of it zero
  CK(cudaMemsetAsync(c->d_Bsum, 0, (size_t)(NG * 3 + 1) * 8, c->stream));
  c->table_groups = NG;
  return 0;
}

static void fill_key_params(tdsfs_ctx* c, KeyParams& p) {
  memset(&p, 0, sizeof p);
  p.n1 = c->n1; p.n2 = c->n2; p.fold = c->fold; p.C2 = c->R2; p.bins2d = c->bins2d; p.R1 = c->R1; p.R2 = c->R2;
  p.ns1 = c->ns1; p.ns2 = c->ns2; p.W1 = c->W1; p.W2 = c->W2;
  p.S = c->S;
  p.G = c->dG; p.cnt = c->dCnt; p.pos = c->dPos; p.flags = c->dFlags; p.fix = c->dFix; p.nfix = c->nfix;
  p.rec = c->d_rec; p.fmt = c->fmt; p.hist = c->d_hist; p.gstride = c->gstride;
  p.chrom_off = c->d_off; p.C = c->C; p.err = c->d_err;
  p.cr = std::min(c->R1, CORNER); p.cc = std::min(c->R2, CORNER);
  p.h1a = std::min(c->R1, H1CAP); p.h1b = std::min(c->R2, H1CAP);
}

extern "C" int tdsfs_background(tdsfs_t* c, int32_t mode, int32_t bg_chrom, int64_t bg_lo, int64_t bg_hi) {
  if (!c) return fail(TDSFS_ERR_ARG, "ctx is NULL");
  if (!c->loaded) return fail(TDSFS_ERR_STATE, "load data first");
  if (mode < TDSFS_BG_NONE || mode > TDSFS_BG_CHROM) return fail(TDSFS_ERR_ARG, "bad background mode %d", mode);
  // bg_chrom = -1: none of this handle's chromosomes is in the background (a rank of a sharded scan that does not own the
  // background chromosome): the single-group histogram is still allocated and zeroed so that it can take part in the sum
  if (mode == TDSFS_BG_CHROM && (bg_chrom < -1 || bg_chrom >= c->C)) return fail(TDSFS_ERR_ARG, "background chromosome %d out of range", bg_chrom);
  CK(cudaSetDevice(c->device));
  NvtxRange nvtx("tdsfs:K1 count kernel (+ window sums)");
  cudaStream_t st = c->stream;
  c->ws_ready = false;  // the records (and any window sums) are rewritten by this pass
  CK(cudaEventRecord(c->ev[EV_BG0], st));
  const int NG = mode == TDSFS_BG_PER_CHROM ? c->C : 1;
  c->gstride = (long long)c->bins2d + c->R1 + c->R2;
  const long long words = c->gstride * NG;
  if (words > c->hist_words) {
    peer_unmap(c);
    c->peer_exported_hist = nullptr;
    dev_free(c->d_hist);
    CKR(dev_alloc(&c->d_hist, words));
    c->hist_words = words;
  }
  CK(cudaMemsetAsync(c->d_hist, 0, (size_t)words * 4, st));
  CK(cudaMemsetAsync(c->d_err, 0, sizeof(int), st));
  c->NG = NG;
  c->bg_mode = mode;
  c->float_bg = false;
  c->poisson_bg = false;
  c->tables_from_exchange = false;
  c->tables_ready = false;
  c->results_ready = false;
  c->per_chrom_scoring = mode == TDSFS_BG_PER_CHROM;

  // record format: 4-byte narrow records when the 2D cell plus two missing-diploid counts fit 32 bits (genotype entry,
  // no half-call fix-ups, no more sample columns than the declared panel); 8-byte wide records otherwise
  c->fmt = RecFmt{0, 0, 0, 0};
  if (c->dG && !c->force_wide && c->nfix == 0 && c->ns1 <= c->n1 && c->ns2 <= c->n2 && !getenv("TDSFS_REC_WIDE")) {
    int b1 = 1, b2 = 1;
    while ((1 << b1) <= 2 * c->n1) ++b1;
    while ((1 << b2) <= 2 * c->n2) ++b2;
    const int md = (32 - b1 - b2) / 2;
    if (md >= 3) c->fmt = RecFmt{1, b1, b2, md};
  }
  KeyParams p;
  fill_key_params(c, p);
  p.bg_lo = bg_lo; p.bg_hi = bg_hi;
  if (bg_lo < 0 || bg_hi < 0) { p.bg_lo = -1; p.bg_hi = -1; }
  p.bg_group = nullptr;
  p.uniform_group = mode == TDSFS_BG_GENOME ? 0 : -1;
  if (mode == TDSFS_BG_PER_CHROM || mode == TDSFS_BG_CHROM) {
    if (c->groups_mode != mode || c->groups_chrom != bg_chrom) {  // upload once per (mode, chromosome)
      std::vector<int32_t> g(c->C), sg(c->C);
      for (int i = 0; i < c->C; ++i) {
        g[i] = mode == TDSFS_BG_PER_CHROM ? i : (i == bg_chrom ? 0 : -1);
        sg[i] = i;
      }
      dev_free(c->d_bg_group);
      dev_free(c->d_score_group);
      CKR(dev_alloc(&c->d_bg_group, c->C));
      CKR(dev_alloc(&c->d_score_group, c->C));
      CK(cudaMemcpyAsync(c->d_bg_group, g.data(), (size_t)c->C * 4, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(c->d_score_group, sg.data(), (size_t)c->C * 4, cudaMemcpyHostToDevice, st));
      CK(cudaStreamSynchronize(st));  // g / sg are stack-lifetime buffers
      c->groups_mode = mode;
      c->groups_chrom = bg_chrom;
    }
    p.bg_group = c->d_bg_group;
  }

  const int hist_bytes = (p.cr * p.cc + p.h1a + p.h1b) * 4;
  if (c->dG) {
    const int RW = c->W1 + c->W2;
    const int blk_bytes = RW * BLK * 4;
    if (blk_bytes > 32 * 1024) {
      // wide rows (> 4096 samples): stream every 32-SNP block as segments of 64 words (8 KB)
      const int seg_words = 64;
      p.tile_blocks = 1;
      p.stage_bytes = seg_words * BLK * 4;
      const int fit = (226 * 1024 - hist_bytes) / (p.stage_bytes + 8);
      p.cwarps = std::min(K1_DEFAULT_WARPS, fit / 2);
      p.nstage = p.cwarps * 2;
      const int smem = p.nstage * p.stage_bytes + p.nstage * 8 + hist_bytes;
      CK(cudaFuncSetAttribute(k1_genotypes_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      for (auto& ch : c->chunks) {
        if (ch.r1 <= ch.r0) continue;
        if (ch.ev) CK(cudaStreamWaitEvent(st, ch.ev, 0));
        p.r0 = ch.r0; p.r1 = ch.r1;
        const long long nblk = (ch.r1 - ch.r0 + BLK - 1) / BLK;
        const int grid = (int)std::min<long long>(nblk, (long long)c->sm_count);
        k1_genotypes_wide<<<grid, K1_DEFAULT_WARPS * 32, smem, st>>>(p, seg_words);
        c->launches++;
      }
    } else {
      // Ring geometry (measured, profiles/README.md "K1 ring geometry"): ONE stage per warp and about 128 KB of tiles in
      // flight per SM.  Rows up to 8 KB per block use two-block tiles; more warps for narrow rows (more per-SNP work per
      // byte), fewer and larger requests for wide rows.  Deeper rings and more bytes in flight are slower on B200.
      // fused kernel (measured, profiles/README.md round 2): it is bound by per-warp instruction latency, not by bytes in
      // flight, so it takes as many warps as fit, with tiles of at most 8 KB halved until the warp limit is reached
      // (config 5: 14 warps x 8 KB, config 4: 24 warps x 3.5 KB); without window sums (an unplanned scan) it keeps the
      // round-1 rule (128 KB in flight)
      // ---- fused scan: a plan for (W, mode) is pending -> the count kernel also leaves every window's background-independent sums
      FusedParams q;
      memset(&q, 0, sizeof q);
      const int hist_words = (p.cr * p.cc + p.h1a + p.h1b + 3) & ~3;
      q.nw1 = (c->n1 + 2) / 2; q.nw2 = (c->n2 + 2) / 2;
      const int tab_words = HASH_SLOTS + ((q.nw1 + q.nw2 + 3) & ~3);
      const int smem_max = 227 * 1024;
      bool fuse = c->plan_W > 0 && c->plan_W <= 0x7FFFFFFFLL && score_small_ok(c->n1, c->n2, c->bins2d) &&
                  !(c->plan_snp && c->plan_W > WCAP);
      auto fit_for = [&](int tile_blocks, bool with_tables) {
        const int stride = tile_blocks * blk_bytes + tile_blocks * BLK * 4;
        return (smem_max - hist_words * 4 - 16) / (stride + 8 + (with_tables ? tab_words * 4 : 0));
      };
      p.tile_blocks = std::max(1, 8192 / blk_bytes);  // one TMA bulk copy per tile
      if (fuse && fit_for(1, true) < 4) fuse = false;  // panel too large for warp-private window tables beside the ring: table scorer
      if (fuse)
        while (p.tile_blocks > 1 && fit_for(p.tile_blocks, true) < K1_CWARPS) p.tile_blocks /= 2;
      else if (blk_bytes <= 8192)
        p.tile_blocks = std::max(2, p.tile_blocks);
      if (const char* e = getenv("TDSFS_K1_TILE")) p.tile_blocks = std::max(1, atoi(e));  // tuning knob: blocks per tile
      p.stage_bytes = p.tile_blocks * blk_bytes;
      const int stage_stride = p.stage_bytes + p.tile_blocks * BLK * 4;
      const int fit = fit_for(p.tile_blocks, fuse);
      if (fit < 1) return fail(TDSFS_ERR_ARG, "row too wide for the count kernel's shared-memory ring");
      const int max_warps = (c->W1 == 32 && c->W2 == 32) ? k1f_max_warps<32, 32>() : K1_CWARPS;  // launch bound of the instantiation
      p.cwarps = fuse ? std::min(fit, max_warps) : std::min(fit, std::max(4, std::min(max_warps, (128 * 1024) / p.stage_bytes)));
      if (const char* e = getenv("TDSFS_K1_WARPS")) p.cwarps = std::max(1, std::min(std::min(max_warps, fit), atoi(e)));  // tuning knob
      int depth = 1;  // stages per warp
      if (const char* e = getenv("TDSFS_K1_DEPTH")) depth = std::max(1, atoi(e));  // tuning knob
      q.wmode = fuse ? (c->plan_snp ? 2 : 1) : 0;
      q.tab_words = fuse ? tab_words : 0;
      if (fuse) {
        const long long ncand = c->cand.off[c->C];
        if (ncand > c->ws_cap) {
          CK(cudaStreamSynchronize(st));
          dev_free(c->d_ws);
          CKR(dev_alloc(&c->d_ws, ncand * 4));
          c->ws_cap = ncand;
        }
        q.W = (uint32_t)c->plan_W;
        q.Wmagic = (uint32_t)std::min<unsigned long long>(0xFFFFFFFFull, (1ull << 32) / (unsigned long long)c->plan_W);
        q.cand_off = c->cand.d_off;
        q.ncand = ncand;
        q.ws = c->d_ws;
        q.dxI = c->d_dxI;
        q.lnI = c->d_lnI;
      } else {
        q.nw1 = q.nw2 = 0;
      }
      q.pos_tma = (((uintptr_t)c->dPos) & 15) == 0 && !getenv("TDSFS_NO_POS_TMA");
      // ring depth: as many stages per warp as asked for and as fit beside the histograms and the window tables
      const int per_warp_fixed = q.tab_words * 4;
      while (depth > 1 && p.cwarps * (depth * (stage_stride + 8) + per_warp_fixed) + hist_words * 4 + 16 > smem_max) --depth;
      p.nstage = p.cwarps * depth;
      const int smem = p.nstage * stage_stride + p.cwarps * q.tab_words * 4 + ((p.nstage + 1) & ~1) * 8 + hist_words * 4;
      if (smem > smem_max) return fail(TDSFS_ERR_ARG, "count kernel geometry needs %d bytes of shared memory (warps %d, depth %d)", smem, p.cwarps, depth);
      // PLAIN instantiation: every per-SNP branch that cannot trigger in the common configuration compiled out
      const bool plain = !c->dFlags && c->nfix == 0 && p.bg_group == nullptr && p.bg_lo < 0 && c->fold && c->fmt.narrow &&
                         c->n1 >= 32 && c->n2 >= 32 && c->n1 <= 1023 && c->n2 <= 1023;
      void (*kern)(FusedParams) = plain ? k1_fused<0, 0, true> : k1_fused<0, 0, false>;
      if (plain && c->W1 == 32 && c->W2 == 32) kern = k1_fused<32, 32, true>;        // 500 + 500 diploids (BASELINE config 5)
      else if (plain && c->W1 == 14 && c->W2 == 14) kern = k1_fused<14, 14, true>;   // 200 + 200 diploids (BASELINE config 4)
      CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      // Tail of the launch: inside tdsfs_step_bp with the peer exchange mapped, a pass that is ONE launch over resident data (the
      // usual case) exchanges the histogram with the other ranks after a grid-wide barrier and builds the ln tables of the
      // background, instead of leaving that to a separate launch.  (Measured: without an exchange, ln tables in the tail only
      // match the separate finalize launch of a replayed graph.)
      const bool one_launch = c->chunks.size() == 1 && !c->chunks[0].ev && c->chunks[0].r1 > c->chunks[0].r0;
      const bool tail = c->want_tail_exchange && one_launch && mode != TDSFS_BG_NONE && NG == 1 && c->peer_ready &&
                        c->d_hist == c->peer_exported_hist && c->gstride == c->peer_words;
      if (tail) {
        CKR(ensure_tables(c, NG));
        q.tail = 1;
        q.gridbar = c->d_gridbar;
        q.tail_timeout = PEER_TIMEOUT_CYCLES;
        q.stamps = c->d_stamps;
        FinParams& f = q.fin;
        f.hist = c->d_hist; f.gstride = c->gstride; f.NG = NG; f.bins2d = c->bins2d; f.R1 = c->R1; f.R2 = c->R2;
        f.n1 = c->n1; f.n2 = c->n2; f.lb2 = c->d_lb2; f.lb1a = c->d_lb1a; f.lb1b = c->d_lb1b; f.Bsum = c->d_Bsum; f.B = c->d_B;
        for (int r = 0; r < PEER_MAX; ++r) { q.peer.hist[r] = c->peer_hist[r]; q.peer.flags[r] = c->peer_flags[r]; }
        q.peer.rank = c->peer_rank; q.peer.world = c->peer_world; q.peer.words = c->peer_words; q.peer.err = c->d_err;
        q.peer.timeout_cycles = PEER_TIMEOUT_CYCLES;
        q.peer.ticket = reinterpret_cast<unsigned int*>(c->d_peer_flags + PEER_MAX);
        q.epoch_mem = c->d_peer_flags + PEER_MAX + 1;
      }
      const long long tile_rows = (long long)p.tile_blocks * BLK;
      for (auto& ch : c->chunks) {
        if (ch.r1 <= ch.r0) continue;
        if (ch.ev) CK(cudaStreamWaitEvent(st, ch.ev, 0));
        p.r0 = ch.r0; p.r1 = ch.r1;
        const long long ntiles = (ch.r1 - ch.r0 + tile_rows - 1) / tile_rows;
        const int grid = (int)std::max<long long>(1, std::min<long long>((ntiles + p.cwarps - 1) / p.cwarps, (long long)c->sm_count));
        q.k = p;
        kern<<<grid, p.cwarps * 32, smem, st>>>(q);
        c->launches++;
      }
      if (fuse) {
        c->fused_W = c->plan_W;
        c->fused_snp = c->plan_snp;
        c->ws_ready = true;
      }
      if (tail) {
        c->tables_ready = true;
        c->tables_from_exchange = true;
        c->fin_timed = false;
      }
    }
  } else {
    p.r0 = 0; p.r1 = c->S;
    const long long ntiles = (c->S + K1C_THREADS - 1) / K1C_THREADS;
    if (ntiles > 0) {
      CK(cudaFuncSetAttribute(k1_counts, cudaFuncAttributeMaxDynamicSharedMemorySize, hist_bytes));
      const int grid = (int)std::min<long long>(ntiles, (long long)c->sm_count * 4);
      k1_counts<<<grid, K1C_THREADS, hist_bytes, st>>>(p);
      c->launches++;
    }
  }
  CK(cudaGetLastError());
  CK(cudaEventRecord(c->ev[EV_K1], st));
  c->keys_ready = true;
  CKR(finish(c));
  if (c->sync) {
    int err = 0;
    CK(cudaMemcpy(&err, c->d_err, sizeof err, cudaMemcpyDeviceToHost));
    if (err & 1) {
      c->keys_ready = false;
      c->ws_ready = false;
      return fail(TDSFS_ERR_RANGE, "an allele count exceeds 2n of the declared panel (n1=%d, n2=%d)", c->n1, c->n2);
    }
    if ((err & 8) && !c->force_wide) {  // a SNP's missing-call counts do not fit the narrow record: redo with wide records
      c->force_wide = true;
      return tdsfs_background(c, mode, bg_chrom, bg_lo, bg_hi);
    }
  }
  return 0;
}

extern "C" int tdsfs_background_device(tdsfs_t* c, void** dev_ptr, int64_t* n_words, int32_t* n_groups) {
  if (!c || !c->keys_ready) return fail(TDSFS_ERR_STATE, "tdsfs_background first");
  CK(cudaSetDevice(c->device));
  c->tables_ready = c->float_bg;  // the caller is about to change the histogram (all-reduce): integer tables are rebuilt by finalize
  c->tables_from_exchange = false;
  if (dev_ptr) *dev_ptr = c->d_hist;
  if (n_words) *n_words = c->gstride * c->NG;
  if (n_groups) *n_groups = c->NG;
  return 0;
}

// ------------------------------------------------------------------------------------------------ peer exchange
struct PeerBlob {  // TDSFS_PEER_BLOB_BYTES
  cudaIpcMemHandle_t hist, flags;
  long long words;
  int rank, world;
  int device, pad;
};
static_assert(sizeof(PeerBlob) <= TDSFS_PEER_BLOB_BYTES, "blob size");

static void peer_unmap(tdsfs_ctx* c) {
  drop_step_graph(c);
  for (int r = 0; r < c->peer_world; ++r) {
    if (r != c->peer_rank) {
      if (c->peer_hist[r]) cudaIpcCloseMemHandle(c->peer_hist[r]);
      if (c->peer_flags[r]) cudaIpcCloseMemHandle(c->peer_flags[r]);
    }
    c->peer_hist[r] = nullptr;
    c->peer_flags[r] = nullptr;
  }
  c->peer_ready = false;
}

extern "C" int tdsfs_peer_export(tdsfs_t* c, int32_t rank, int32_t world, void* blob) {
  if (!c || !blob) return fail(TDSFS_ERR_ARG, "NULL argument");
  if (world < 1 || world > PEER_MAX || rank < 0 || rank >= world) return fail(TDSFS_ERR_ARG, "rank %d / world %d out of range (max %d)", rank, world, PEER_MAX);
  if (!c->keys_ready || !c->d_hist) return fail(TDSFS_ERR_STATE, "tdsfs_background first (the histogram must exist)");
  if (c->NG != 1) return fail(TDSFS_ERR_STATE, "the peer exchange needs a single background group (TDSFS_BG_GENOME / _CHROM)");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  peer_unmap(c);
  if (!c->d_peer_flags) CKR(dev_alloc(&c->d_peer_flags, PEER_MAX + 2));  // flags, the reduce kernel's CTA counter, the epoch
  CK(cudaMemset(c->d_peer_flags, 0, (PEER_MAX + 2) * sizeof(unsigned long long)));
  c->peer_rank = rank;
  c->peer_world = world;
  c->peer_words = c->gstride;
  c->peer_exported_hist = c->d_hist;
  PeerBlob b;
  memset(&b, 0, sizeof b);
  CK(cudaIpcGetMemHandle(&b.hist, c->d_hist));
  CK(cudaIpcGetMemHandle(&b.flags, c->d_peer_flags));
  b.words = c->peer_words; b.rank = rank; b.world = world; b.device = c->device;
  memset(blob, 0, TDSFS_PEER_BLOB_BYTES);
  memcpy(blob, &b, sizeof b);
  return 0;
}

extern "C" int tdsfs_peer_import(tdsfs_t* c, const void* blobs) {
  if (!c || !blobs) return fail(TDSFS_ERR_ARG, "NULL argument");
  if (c->peer_world < 1 || !c->peer_exported_hist) return fail(TDSFS_ERR_STATE, "tdsfs_peer_export first");
  CK(cudaSetDevice(c->device));
  for (int r = 0; r < c->peer_world; ++r) {
    PeerBlob b;
    memcpy(&b, (const char*)blobs + (size_t)r * TDSFS_PEER_BLOB_BYTES, sizeof b);
    if (b.rank != r || b.world != c->peer_world) { peer_unmap(c); return fail(TDSFS_ERR_ARG, "blob %d is from rank %d of %d", r, b.rank, b.world); }
    if (b.words != c->peer_words) { peer_unmap(c); return fail(TDSFS_ERR_ARG, "rank %d holds a histogram of %lld words, this rank %lld: panels differ", r, b.words, c->peer_words); }
    if (r == c->peer_rank) {
      c->peer_hist[r] = c->d_hist;
      c->peer_flags[r] = c->d_peer_flags;
      continue;
    }
    void *ph = nullptr, *pf = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ph, b.hist, cudaIpcMemLazyEnablePeerAccess);
    if (e == cudaSuccess) e = cudaIpcOpenMemHandle(&pf, b.flags, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      if (ph) cudaIpcCloseMemHandle(ph);
      peer_unmap(c);
      cudaGetLastError();
      return fail(TDSFS_ERR_CUDA, "cannot map the histogram of rank %d (device %d): %s", r, b.device, cudaGetErrorString(e));
    }
    c->peer_hist[r] = (uint32_t*)ph;
    c->peer_flags[r] = (unsigned long long*)pf;
  }
  c->peer_ready = true;
  drop_step_graph(c);
  return 0;
}

// All-reduce of the background AND the ln tables in one launch (k_peer_reduce_finalize); a later tdsfs_finalize_background
// is then a no-op.
extern "C" int tdsfs_peer_reduce_finalize(tdsfs_t* c) {
  if (!c || !c->peer_ready) return fail(TDSFS_ERR_STATE, "tdsfs_peer_export / tdsfs_peer_import first");
  if (!c->keys_ready) return fail(TDSFS_ERR_STATE, "tdsfs_background first");
  if (c->d_hist != c->peer_exported_hist || c->NG != 1 || c->gstride != c->peer_words)
    return fail(TDSFS_ERR_STATE, "the histogram changed since tdsfs_peer_export (panel or background mode): export again");
  CK(cudaSetDevice(c->device));
  NvtxRange nvtx("tdsfs:exchange + finalize (one launch)");
  cudaStream_t st = c->stream;
  CKR(ensure_tables(c, 1));
  PeerFinParams q;
  memset(&q, 0, sizeof q);
  for (int r = 0; r < PEER_MAX; ++r) { q.x.hist[r] = c->peer_hist[r]; q.x.flags[r] = c->peer_flags[r]; }
  q.x.rank = c->peer_rank; q.x.world = c->peer_world; q.x.words = c->peer_words; q.x.err = c->d_err;
  q.x.timeout_cycles = PEER_TIMEOUT_CYCLES;
  q.x.ticket = reinterpret_cast<unsigned int*>(c->d_peer_flags + PEER_MAX);
  q.epoch_mem = c->d_peer_flags + PEER_MAX + 1;
  FinParams& f = q.f;
  f.hist = c->d_hist; f.gstride = c->gstride; f.NG = 1; f.bins2d = c->bins2d; f.R1 = c->R1; f.R2 = c->R2;
  f.n1 = c->n1; f.n2 = c->n2; f.lb2 = c->d_lb2; f.lb1a = c->d_lb1a; f.lb1b = c->d_lb1b; f.Bsum = c->d_Bsum; f.B = c->d_B;
  const int grid = (int)std::max(1, std::min(c->sm_count, (c->bins2d + 255) / 256));
  CK(cudaEventRecord(c->ev[EV_X0], st));
  k_peer_reduce_finalize<<<grid, 256, 0, st>>>(q);
  CK(cudaEventRecord(c->ev[EV_X1], st));
  c->x_timed = true;
  c->launches += 1;
  CK(cudaGetLastError());
  c->tables_ready = true;
  c->tables_from_exchange = true;
  c->float_bg = false;
  c->fin_timed = false;  // no separate finalize launch to time
  return finish(c);
}

// the exchange always builds the ln tables in the same launch (include/tdsfs.h)
extern "C" int tdsfs_peer_allreduce_background(tdsfs_t* c) { return tdsfs_peer_reduce_finalize(c); }

extern "C" int tdsfs_peer_close(tdsfs_t* c) {
  if (!c) return fail(TDSFS_ERR_ARG, "ctx is NULL");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  peer_unmap(c);
  c->peer_exported_hist = nullptr;
  c->peer_world = 0;
  c->peer_rank = -1;
  return 0;
}

extern "C" int tdsfs_get_background(tdsfs_t* c, int32_t group, uint64_t* s2, uint64_t* s1a, uint64_t* s1b) {
  if (!c || !c->keys_ready) return fail(TDSFS_ERR_STATE, "tdsfs_background first");
  if (group < 0 || group >= c->NG) return fail(TDSFS_ERR_ARG, "group %d out of range", group);
  CK(cudaSetDevice(c->device));
  std::vector<uint32_t> h((size_t)c->gstride);
  CK(cudaMemcpyAsync(h.data(), c->d_hist + (long long)group * c->gstride, (size_t)c->gstride * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (s2) for (int i = 0; i < c->bins2d; ++i) s2[i] = h[i];
  if (s1a) for (int i = 0; i < c->R1; ++i) s1a[i] = h[c->bins2d + i];
  if (s1b) for (int i = 0; i < c->R2; ++i) s1b[i] = h[c->bins2d + c->R1 + i];
  return 0;
}

extern "C" int tdsfs_set_background(tdsfs_t* c, const double* b2d, const double* b1a, const double* b1b) {
  if (!c || !b2d || !b1a || !b1b) return fail(TDSFS_ERR_ARG, "NULL argument");
  if (!c->bins2d) return fail(TDSFS_ERR_STATE, "tdsfs_set_panel first");
  CK(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  CKR(ensure_tables(c, 1));
  // interior totals summed on the host in index order, as the reference's sum(counts_bg) does (:665, :517)
  double B[6] = {0, 0, 0, 0, 0, 0};
  for (int k = 1; k < c->bins2d - 1; ++k) B[0] += b2d[k];
  for (int k = 1; k <= c->n1 - 1; ++k) B[1] += b1a[k];
  for (int k = 1; k <= c->n2 - 1; ++k) B[2] += b1b[k];
  for (int q = 0; q < 3; ++q) B[3 + q] = B[q] > 0.0 ? log(B[q]) : (B[q] == 0.0 ? -INFINITY : NAN);
  void* tmp = nullptr;  // pooled staging buffer for the three value vectors
  CKR(pool_get(&c->pool_tmp, &c->cap_tmp, ((size_t)c->bins2d + c->n1 + 1 + c->n2 + 1) * sizeof(double), &tmp));
  double *t2 = (double*)tmp, *t1a = t2 + c->bins2d, *t1b = t1a + c->n1 + 1;
  CK(cudaMemcpyAsync(t2, b2d, (size_t)c->bins2d * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(t1a, b1a, (size_t)(c->n1 + 1) * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(t1b, b1b, (size_t)(c->n2 + 1) * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(c->d_B, B, sizeof B, cudaMemcpyHostToDevice, st));
  k_log_table<<<std::min(1024, (c->bins2d + 255) / 256), 256, 0, st>>>(t2, c->d_lb2, c->bins2d);
  k_log_table<<<1, 256, 0, st>>>(t1a, c->d_lb1a, c->n1 + 1);
  k_log_table<<<1, 256, 0, st>>>(t1b, c->d_lb1b, c->n2 + 1);
  c->launches += 3;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(st));  // the host vectors are the caller's: they may change after the call returns
  c->float_bg = true;
  c->poisson_bg = false;
  c->per_chrom_scoring = false;
  c->tables_ready = true;
  c->results_ready = false;
  return 0;
}

extern "C" int tdsfs_set_poisson_background(tdsfs_t* c, const double* q2d) {
  if (!c || !q2d) return fail(TDSFS_ERR_ARG, "NULL argument");
  if (!c->bins2d) return fail(TDSFS_ERR_STATE, "tdsfs_set_panel first");
  CK(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  CKR(ensure_tables(c, 1));
  std::vector<double> lq((size_t)c->bins2d);
  double n = 0, sum = 0, lnsum = 0;
  for (int k = 0; k < c->bins2d; ++k) {
    const double q = q2d[k];
    if (q != 0.0) {  // a bin with a zero expectation is skipped by the score (twoDSFS.py:364)
      n += 1; sum += q; lnsum += log(q);
      lq[k] = log(q);
    } else {
      lq[k] = -INFINITY;
    }
  }
  CK(cudaMemcpyAsync(c->d_lb2, lq.data(), (size_t)c->bins2d * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(c->d_lb1a, 0, (size_t)(c->n1 + 1) * 8, st));
  CK(cudaMemsetAsync(c->d_lb1b, 0, (size_t)(c->n2 + 1) * 8, st));
  CK(cudaStreamSynchronize(st));
  c->pq_n = n; c->pq_sum = sum; c->pq_lnsum = lnsum;
  c->float_bg = true;
  c->poisson_bg = true;
  c->per_chrom_scoring = false;
  c->tables_ready = true;
  c->results_ready = false;
  return 0;
}

extern "C" int tdsfs_finalize_background(tdsfs_t* c) {
  if (!c) return fail(TDSFS_ERR_ARG, "ctx is NULL");
  if (c->float_bg) return 0;  // tables were built by tdsfs_set_background
  if (c->tables_from_exchange && c->tables_ready) return 0;  // ... or by tdsfs_peer_reduce_finalize
  if (!c->keys_ready || c->bg_mode == TDSFS_BG_NONE) return fail(TDSFS_ERR_STATE, "no integer background to finalize");
  CK(cudaSetDevice(c->device));
  NvtxRange nvtx("tdsfs:finalize (ln tables)");
  cudaStream_t st = c->stream;
  CK(cudaEventRecord(c->ev[EV_FIN0], st));
  CKR(ensure_tables(c, c->NG));
  FinParams f;
  memset(&f, 0, sizeof f);
  f.hist = c->d_hist; f.gstride = c->gstride; f.NG = c->NG; f.bins2d = c->bins2d; f.R1 = c->R1; f.R2 = c->R2;
  f.n1 = c->n1; f.n2 = c->n2; f.lb2 = c->d_lb2; f.lb1a = c->d_lb1a; f.lb1b = c->d_lb1b; f.Bsum = c->d_Bsum; f.B = c->d_B;
  // one bin per thread up to four CTAs per SM (measured: ~8 bins per thread with a smaller grid is slower for the 401 x 401 spectrum)
  dim3 grid((unsigned)std::max(1, std::min(c->sm_count * 4, (c->bins2d + 255) / 256)), (unsigned)c->NG);
  k_finalize_counts<<<grid, 256, 0, st>>>(f);
  c->launches += 1;
  CK(cudaGetLastError());
  CK(cudaEventRecord(c->ev[EV_FIN1], st));
  c->tables_ready = true;
  c->fin_timed = true;
  CKR(finish(c));
  return 0;
}

// ------------------------------------------------------------------------------------------------ scans
static int candidates(tdsfs_ctx* c, long long W, bool snp_mode, std::vector<long long>& off) {
  off.assign(c->C + 1, 0);
  for (int i = 0; i < c->C; ++i) {
    long long n = 0;
    const long long sc = c->h_off[i + 1] - c->h_off[i];
    if (sc > 0) n = snp_mode ? sc / W : (std::max<long long>(c->h_last[i] - 1, 0) / W + 1);
    off[i + 1] = off[i] + n;
  }
  if (off[c->C] > 0x7FFFFFF0LL) return fail(TDSFS_ERR_ARG, "too many candidate windows (%lld)", off[c->C]);
  return 0;
}

static int count_candidates(tdsfs_ctx* c, long long W, bool snp_mode, int64_t* n) {
  if (!c || !n || W < 1) return fail(TDSFS_ERR_ARG, "bad argument");
  if (!c->dPos) return fail(TDSFS_ERR_STATE, "load data first");
  std::vector<long long> off;
  CKR(candidates(c, W, snp_mode, off));
  *n = off[c->C];
  return 0;
}
extern "C" int tdsfs_candidates_bp(tdsfs_t* c, int64_t W, int64_t* n) { return count_candidates(c, W, false, n); }
extern "C" int tdsfs_candidates_snp(tdsfs_t* c, int64_t N, int64_t* n) { return count_candidates(c, N, true, n); }

// The offsets of (W, mode) in k, uploaded on stream st when they change.
static int cached_candidates(tdsfs_ctx* c, CandCache& k, long long W, bool snp_mode, cudaStream_t st) {
  if (k.holds(W, snp_mode)) return 0;
  k.W = -1;  // until the device copy matches
  CKR(candidates(c, W, snp_mode, k.off));
  dev_free(k.d_off);
  CKR(dev_alloc(&k.d_off, c->C + 1));
  CK(cudaMemcpyAsync(k.d_off, k.off.data(), (size_t)(c->C + 1) * 8, cudaMemcpyHostToDevice, st));
  k.W = W;
  k.snp = snp_mode;
  return 0;
}

static int ensure_windows(tdsfs_ctx* c, long long n) {
  if (n <= c->cand_cap) return 0;
  // growing: a previous asynchronous scan may still be using the old arrays
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaStreamSynchronize(c->plan_stream));
  dev_free(c->d_wlo); dev_free(c->d_whi); dev_free(c->d_wchrom); dev_free(c->d_large); dev_free(c->d_wstart); dev_free(c->d_wend);
  dev_free(c->r_count); dev_free(c->r_n2); dev_free(c->r_n1a); dev_free(c->r_n1b); dev_free(c->r_T2); dev_free(c->r_T1a);
  dev_free(c->r_T1b); dev_free(c->r_flags);
  CKR(dev_alloc(&c->d_wlo, n)); CKR(dev_alloc(&c->d_whi, n)); CKR(dev_alloc(&c->d_wchrom, n)); CKR(dev_alloc(&c->d_large, n));
  CKR(dev_alloc(&c->d_wstart, n)); CKR(dev_alloc(&c->d_wend, n));
  CKR(dev_alloc(&c->r_count, n)); CKR(dev_alloc(&c->r_n2, n)); CKR(dev_alloc(&c->r_n1a, n)); CKR(dev_alloc(&c->r_n1b, n));
  CKR(dev_alloc(&c->r_T2, n)); CKR(dev_alloc(&c->r_T1a, n)); CKR(dev_alloc(&c->r_T1b, n)); CKR(dev_alloc(&c->r_flags, n));
  c->cand_cap = n;
  return 0;
}

// n windows of one per-window result: host destination (NULL: not wanted), device source
struct Column {
  template <typename H, typename D>
  Column(H* dst, const D* src) : dst(dst), src(src), size(sizeof(D)) { static_assert(sizeof(H) == sizeof(D), "element size"); }
  void* dst;
  const void* src;
  size_t size;
};

// Copies n windows of each wanted column to the host on the handle's stream (its device current), then waits for them.
static int fetch_columns(tdsfs_ctx* c, long long n, std::initializer_list<Column> cols, int64_t* n_windows) {
  for (const Column& k : cols)
    if (k.dst && n) CK(cudaMemcpyAsync(k.dst, k.src, (size_t)n * k.size, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (n_windows) *n_windows = n;
  return 0;
}

extern "C" int tdsfs_fetch_results(tdsfs_t* c, tdsfs_result_t* out, int64_t cap, int64_t* n_windows) {
  if (!c || !out) return fail(TDSFS_ERR_ARG, "NULL argument");
  if (!c->results_ready) return fail(TDSFS_ERR_STATE, "no scan results");
  if (cap < c->ncand) return fail(TDSFS_ERR_ARG, "result capacity %lld < %lld candidate windows", (long long)cap, c->ncand);
  CK(cudaSetDevice(c->device));
  int err = 0;  // read in the same round trip as the results
  CK(cudaMemcpyAsync(&err, c->d_err, sizeof err, cudaMemcpyDeviceToHost, c->stream));
  CKR(fetch_columns(c, c->ncand, {{out->chrom, c->d_wchrom}, {out->start, c->d_wstart}, {out->end, c->d_wend},
                                  {out->snp_count, c->r_count}, {out->n2d, c->r_n2}, {out->n1d_p1, c->r_n1a},
                                  {out->n1d_p2, c->r_n1b}, {out->T2D, c->r_T2}, {out->T1D_p1, c->r_T1a},
                                  {out->T1D_p2, c->r_T1b}, {out->flags, c->r_flags}}, n_windows));
  return deferred_error(c, err);
}

// candidate list of (W, mode) on the device + K2 launch on stream `st`
static int ensure_candidates(tdsfs_ctx* c, long long W, bool snp_mode, cudaStream_t st) {
  if (!c->cand.holds(W, snp_mode)) c->ws_ready = false;  // the count kernel's window sums are of other windows
  CKR(cached_candidates(c, c->cand, W, snp_mode, st));
  return ensure_windows(c, c->cand.off[c->C]);
}

static int launch_bounds(tdsfs_ctx* c, long long W, bool snp_mode, cudaStream_t st) {
  CKR(ensure_candidates(c, W, snp_mode, st));
  const long long ncand = c->cand.off[c->C];
  if (ncand > 0) {
    CK(cudaMemsetAsync(c->d_nlarge, 0, sizeof(int), st));
    WinParams w;
    w.pos = c->dPos; w.chrom_off = c->d_off; w.cand_off = c->cand.d_off; w.C = c->C; w.W = W; w.ncand = ncand;
    w.wlo = c->d_wlo; w.whi = c->d_whi; w.wchrom = c->d_wchrom; w.wstart = c->d_wstart; w.wend = c->d_wend;
    w.large = c->d_large; w.nlarge = c->d_nlarge;
    w.r_count = c->r_count; w.r_flags = c->r_flags;
    w.wcap = score_small_ok(c->n1, c->n2, c->bins2d) && score_group_smem_words(c->n1, c->n2) * 4 <= 200 * 1024 ? WCAP : 0;
    const int g2 = (int)((ncand + 255) / 256);
    if (snp_mode) k2_bounds_snp<<<g2, 256, 0, st>>>(w); else k2_bounds_bp<<<g2, 256, 0, st>>>(w);
    c->launches++;
    CK(cudaGetLastError());
  }
  return 0;
}

// Window boundaries depend on positions only: launch K2 on a side stream now so that it overlaps the count kernel and the
// background all-reduce; the next scan of the same (size, mode) waits for it instead of launching K2 itself.
static int plan(tdsfs_ctx* c, long long W, bool snp_mode) {
  if (!c || W < 1) return fail(TDSFS_ERR_ARG, "bad argument");
  if (!c->dPos) return fail(TDSFS_ERR_STATE, "load data first");
  CK(cudaSetDevice(c->device));
  NvtxRange nvtx("tdsfs:K2 window boundaries (side stream)");
  CKR(ensure_candidates(c, W, snp_mode, c->stream));     // the fused count kernel (main stream) reads the candidate offsets too
  CK(cudaEventRecord(c->ev_fork, c->stream));            // after everything queued so far (previous scan reads the old plan)
  CK(cudaStreamWaitEvent(c->plan_stream, c->ev_fork, 0));
  CK(cudaEventRecord(c->ev_plan0, c->plan_stream));
  CKR(launch_bounds(c, W, snp_mode, c->plan_stream));
  CK(cudaEventRecord(c->ev_plan, c->plan_stream));
  c->plan_W = W;
  c->plan_snp = snp_mode;
  c->results_ready = false;
  return 0;
}
extern "C" int tdsfs_plan_bp(tdsfs_t* c, int64_t W) { return plan(c, W, false); }
extern "C" int tdsfs_plan_snp(tdsfs_t* c, int64_t N) { return plan(c, N, true); }

static int scan(tdsfs_ctx* c, long long W, bool snp_mode, tdsfs_result_t* out, int64_t cap, int64_t* n_windows, bool poisson = false) {
  if (!c || W < 1) return fail(TDSFS_ERR_ARG, "bad argument");
  if (poisson != c->poisson_bg) return fail(TDSFS_ERR_STATE, poisson ? "tdsfs_set_poisson_background first" : "the tables hold a Poisson background: tdsfs_scan_poisson_bp, or set a likelihood background");
  if (poisson && c->fold) return fail(TDSFS_ERR_STATE, "the Poisson score works on the unfolded spectrum: tdsfs_set_panel(..., fold = 0)");
  if (!c->keys_ready) return fail(TDSFS_ERR_STATE, "tdsfs_background first");
  if (!c->tables_ready) return fail(TDSFS_ERR_STATE, "tdsfs_finalize_background / tdsfs_set_background first");
  CK(cudaSetDevice(c->device));
  NvtxRange nvtx("tdsfs:K3 window statistics");
  cudaStream_t st = c->stream;
  const bool planned = c->plan_W == W && c->plan_snp == (int)snp_mode;
  c->plan_W = -1;
  CK(cudaEventRecord(c->ev[EV_SC0], st));
  if (planned) CK(cudaStreamWaitEvent(st, c->ev_plan, 0));   // K2 already ran (or is running) on the side stream
  else CKR(launch_bounds(c, W, snp_mode, st));
  c->planned_last = planned;
  const long long ncand = c->cand.off[c->C];
  if (out && cap < ncand) return fail(TDSFS_ERR_ARG, "result capacity %lld < %lld candidate windows", (long long)cap, ncand);
  c->ncand = ncand;
  CK(cudaEventRecord(c->ev[EV_K2], st));
  if (ncand > 0) {
    ScoreParams s;
    memset(&s, 0, sizeof s);
    s.rec = c->d_rec; s.flags = c->dFlags; s.wlo = c->d_wlo; s.whi = c->d_whi; s.wchrom = c->d_wchrom;
    s.score_group = c->per_chrom_scoring ? c->d_score_group : nullptr;
    s.ncand = ncand; s.n1 = c->n1; s.n2 = c->n2; s.bins2d = c->bins2d; s.snp_mode = snp_mode;
    s.lb2 = c->d_lb2; s.lb1a = c->d_lb1a; s.lb1b = c->d_lb1b; s.B = c->d_B; s.lnI = c->d_lnI;
    s.r_count = c->r_count; s.r_n2 = c->r_n2; s.r_n1a = c->r_n1a; s.r_n1b = c->r_n1b; s.r_T2 = c->r_T2; s.r_T1a = c->r_T1a;
    s.r_T1b = c->r_T1b; s.r_flags = c->r_flags; s.large = c->d_large; s.nlarge = c->d_nlarge;
    s.fmt = c->fmt; s.C2 = c->R2;
    s.poisson = poisson ? 1 : 0; s.pq_n = c->pq_n; s.pq_sum = c->pq_sum; s.pq_lnsum = c->pq_lnsum;
    const long long sstride = (long long)c->bins2d + c->n1 + 1 + c->n2 + 1;
    if (!c->d_scratch) {  // dense scratch of the large-window path, one slab per CTA
      c->large_ctas = (int)std::max<long long>(8, std::min<long long>(2 * c->sm_count, (256LL << 20) / (sstride * 4)));
      CKR(dev_alloc(&c->d_scratch, sstride * c->large_ctas));
      CK(cudaMemsetAsync(c->d_scratch, 0, (size_t)(sstride * c->large_ctas) * 4, st));
    }
    s.scratch = c->d_scratch;
    const int gwords = score_group_smem_words(c->n1, c->n2);
    if (c->ws_ready && c->fused_W == W && c->fused_snp == (int)snp_mode && !poisson) {
      // fused scan: the count kernel left every small window's background-independent sums; one launch gathers ln b over
      // the records, finishes the statistics and scores the large windows
      FinishParams f;
      memset(&f, 0, sizeof f);
      f.s = s;
      f.ws = c->d_ws;
      const size_t tab_bytes = ((size_t)CORNER * CORNER + 2 * c->n1 + 1 + 2 * c->n2 + 1) * sizeof(double);
      f.use_smem = c->fmt.narrow && !c->per_chrom_scoring && c->R1 >= CORNER && c->R2 >= CORNER && tab_bytes <= 96 * 1024;
      f.large_ctas = c->large_ctas;
      const int smem = f.use_smem ? (int)tab_bytes : 0;
      void (*fk)(FinishParams) = k3_finish;
      CK(cudaFuncSetAttribute(fk, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      int occ = 1;
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fk, 256, smem));
      const int grid = (int)std::max<long long>(1, std::min<long long>((ncand + 7) / 8, (long long)c->sm_count * std::max(1, occ)));
      fk<<<grid, 256, smem, st>>>(f);
      c->launches++;
      c->last_fused = true;
      CK(cudaEventRecord(c->ev[EV_K3S], st));
      CK(cudaEventRecord(c->ev[EV_K3L], st));
      CK(cudaGetLastError());
    } else {
    c->last_fused = false;
    // small windows: groups of G warps per window over shared-memory tables (skipped for panels beyond their limits:
    // K2 then lists every window as "large")
    if (score_small_ok(c->n1, c->n2, c->bins2d) && gwords * 4 <= 200 * 1024) {
      // one warp per window when every resident warp gets many windows; two warps per window for small scans
      // (a rank of an 8-GPU run: ~4 windows per warp -> finer granularity evens out the tail; measured 0.135 -> 0.122 ms)
      int G = c->score_group_warps;
      if (ncand < 16LL * c->sm_count * 24) G = std::max(G, 2);
      if (const char* e = getenv("TDSFS_SCORE_G")) G = atoi(e) >= 4 ? 4 : (atoi(e) >= 2 ? 2 : 1);  // tuning knob
      if (poisson) G = 1;
      while (G < SCORE_WARPS && (SCORE_WARPS / G) * gwords * 4 > 200 * 1024) G *= 2;  // fewer, wider groups for big panels
      const int smem = (SCORE_WARPS / G) * gwords * 4;
      const bool extra = snp_mode || c->dFlags != nullptr || poisson;
#define TDSFS_PICK(K, E) (G >= 8 ? K<8, E> : (G == 4 ? K<4, E> : (G == 2 ? K<2, E> : K<1, E>)))
      void (*sk)(ScoreParams) = extra ? TDSFS_PICK(k3_score_small, true) : TDSFS_PICK(k3_score_small, false);
#undef TDSFS_PICK
      CK(cudaFuncSetAttribute(sk, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      int occ = 1;
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, sk, SCORE_WARPS * 32, smem));
      occ = std::max(1, occ);
      const long long want = (ncand + (SCORE_WARPS / G) - 1) / (SCORE_WARPS / G);
      const int grid = (int)std::min<long long>(want, (long long)c->sm_count * occ);
      if (!c->d_work) {
        CKR(dev_alloc(&c->d_work, 1));
        CK(cudaMemsetAsync(c->d_work, 0, 8, st));
        c->work_base = 0;
      }
      s.work = c->d_work;
      s.work_base = c->work_base;
      c->work_base += (unsigned long long)ncand + (unsigned long long)grid * (SCORE_WARPS / G);
      sk<<<grid, SCORE_WARPS * 32, smem, st>>>(s);
      c->launches++;
    }
    CK(cudaEventRecord(c->ev[EV_K3S], st));
    // large windows: one CTA each over dense scratch
    k3_score_large<<<c->large_ctas, LARGE_THREADS, 0, st>>>(s);
    c->launches++;
    CK(cudaEventRecord(c->ev[EV_K3L], st));
    CK(cudaGetLastError());
    }
  } else {
    CK(cudaEventRecord(c->ev[EV_K3S], st));
    CK(cudaEventRecord(c->ev[EV_K3L], st));
  }
  c->results_ready = true;
  if (out) {
    CKR(tdsfs_fetch_results(c, out, cap, n_windows));
  } else {
    if (n_windows) *n_windows = ncand;
    CKR(finish(c));
  }
  return 0;
}

extern "C" int tdsfs_scan_bp(tdsfs_t* c, int64_t W, tdsfs_result_t* out, int64_t cap, int64_t* n) { return scan(c, W, false, out, cap, n); }
extern "C" int tdsfs_scan_snp(tdsfs_t* c, int64_t N, tdsfs_result_t* out, int64_t cap, int64_t* n) { return scan(c, N, true, out, cap, n); }
extern "C" int tdsfs_scan_poisson_bp(tdsfs_t* c, int64_t W, tdsfs_result_t* out, int64_t cap, int64_t* n) { return scan(c, W, false, out, cap, n, true); }

// Synchronise and surface deferred device-side errors (range check of the count kernel).
extern "C" int tdsfs_check(tdsfs_t* c) {
  if (!c) return fail(TDSFS_ERR_ARG, "ctx is NULL");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  int err = 0;
  CK(cudaMemcpy(&err, c->d_err, sizeof err, cudaMemcpyDeviceToHost));
  return deferred_error(c, err);
}

extern "C" int tdsfs_run_bp(tdsfs_t* c, int32_t bg_mode, int64_t W, tdsfs_result_t* out, int64_t cap, int64_t* n) {
  if (!c) return fail(TDSFS_ERR_ARG, "ctx is NULL");
  const bool was_sync = c->sync;
  c->sync = false;  // at most one synchronisation, at the end of the whole pass
  int r = plan(c, W, false);  // K2 on the side stream, concurrent with the count kernel
  if (!r) r = tdsfs_background(c, bg_mode, 0, -1, -1);
  if (!r) r = tdsfs_finalize_background(c);
  if (!r) r = scan(c, W, false, out, cap, n);
  if (!r && (was_sync || out)) r = tdsfs_check(c);  // fully asynchronous otherwise: the caller synchronises and calls tdsfs_check
  if (r == TDSFS_ERR_RETRY) {  // a SNP did not fit the 4-byte record: the handle switched to 8-byte records, run the pass again
    r = plan(c, W, false);
    if (!r) r = tdsfs_background(c, bg_mode, 0, -1, -1);
    if (!r) r = tdsfs_finalize_background(c);
    if (!r) r = scan(c, W, false, out, cap, n);
    if (!r) r = tdsfs_check(c);
  }
  c->sync = was_sync;
  return r;
}

// One whole ASYNCHRONOUS pass on the handle's stream: window plan (side stream) -> count kernel -> exchange + ln tables (one
// launch when the peer exchange is mapped, else finalize) -> finish kernel.  The second call with the same arguments on the
// same data captures the pass as a CUDA graph; later calls replay it (one launch instead of ~10 API calls, and the gaps
// between dependent kernels shrink).  Results stay on the device (tdsfs_fetch_results); errors surface in tdsfs_check.
static int step_eager(tdsfs_ctx* c, int32_t bg_mode, int64_t W) {
  CKR(plan(c, W, false));
  const bool exchange = c->peer_ready && (bg_mode == TDSFS_BG_GENOME || bg_mode == TDSFS_BG_CHROM);
  c->want_tail_exchange = exchange;  // the count kernel's tail exchanges the histogram and builds the tables when it can
  const int r = tdsfs_background(c, bg_mode, 0, -1, -1);
  c->want_tail_exchange = false;
  CKR(r);
  if (!(c->tables_ready && c->tables_from_exchange)) {
    if (exchange && c->NG == 1) CKR(tdsfs_peer_reduce_finalize(c));
    else CKR(tdsfs_finalize_background(c));
  }
  return scan(c, W, false, nullptr, 0, nullptr);
}

extern "C" int tdsfs_step_bp(tdsfs_t* c, int32_t bg_mode, int64_t W) {
  if (!c) return fail(TDSFS_ERR_ARG, "ctx is NULL");
  if (!c->loaded) return fail(TDSFS_ERR_STATE, "load data first");
  CK(cudaSetDevice(c->device));
  const bool was_sync = c->sync;
  c->sync = false;
  int r = 0;
  bool device_resident = true;
  for (auto& ch : c->chunks) if (ch.ev) device_resident = false;  // a host upload in flight is not part of a replayable pass
  if (c->step_exec && c->step_gen == c->generation && c->step_W == W && c->step_mode == bg_mode) {
    NvtxRange nvtx("tdsfs:step (graph replay)");
    cudaError_t e = cudaGraphLaunch(c->step_exec, c->stream);
    if (e != cudaSuccess) r = fail(TDSFS_ERR_CUDA, "cudaGraphLaunch failed: %s", cudaGetErrorString(e));
    c->launches += c->step_launches;
  } else if (!c->step_graphs_off && device_resident && !getenv("TDSFS_NO_GRAPH") && c->warm_gen == c->generation && c->warm_W == W &&
             c->warm_mode == bg_mode) {
    // the previous call ran the same pass eagerly (every buffer is allocated): capture this one
    const long long l0 = c->launches;
    cudaGraph_t graph = nullptr;
    cudaError_t e = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeRelaxed);
    if (e == cudaSuccess) {
      r = step_eager(c, bg_mode, W);
      e = cudaStreamEndCapture(c->stream, &graph);
      if (!r && e == cudaSuccess && graph) e = cudaGraphInstantiate(&c->step_exec, graph, 0);
      if (graph) cudaGraphDestroy(graph);
    }
    if (r || e != cudaSuccess || !c->step_exec) {  // capture not possible here: stay eager
      cudaGetLastError();
      if (c->step_exec) { cudaGraphExecDestroy(c->step_exec); c->step_exec = nullptr; }
      c->step_graphs_off = true;
      r = step_eager(c, bg_mode, W);
    } else {
      c->step_gen = c->generation; c->step_W = W; c->step_mode = bg_mode;
      c->step_launches = c->launches - l0;
      e = cudaGraphLaunch(c->step_exec, c->stream);
      if (e != cudaSuccess) r = fail(TDSFS_ERR_CUDA, "cudaGraphLaunch failed: %s", cudaGetErrorString(e));
    }
  } else {
    r = step_eager(c, bg_mode, W);
    c->warm_gen = c->generation; c->warm_W = W; c->warm_mode = bg_mode;
  }
  c->sync = was_sync;
  return r;
}

extern "C" int tdsfs_window_spectra(tdsfs_t* c, int64_t window, uint64_t* s2, uint64_t* s1a, uint64_t* s1b) {
  if (!c || !c->results_ready) return fail(TDSFS_ERR_STATE, "scan first");
  if (window < 0 || window >= c->ncand) return fail(TDSFS_ERR_ARG, "window %lld out of range", (long long)window);
  CK(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  int32_t lo, hi;
  CK(cudaMemcpyAsync(&lo, c->d_wlo + window, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&hi, c->d_whi + window, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const long long words = (long long)c->bins2d + c->R1 + c->R2;
  uint32_t* d = nullptr;
  CKR(dev_alloc(&d, words));
  CK(cudaMemsetAsync(d, 0, (size_t)words * 4, st));
  if (hi > lo) {
    KeyParams kp;
    fill_key_params(c, kp);
    k_window_hist<<<std::min(1024, (hi - lo + 255) / 256), 256, 0, st>>>(kp, lo, hi, d, d + c->bins2d, d + c->bins2d + c->R1);
    c->launches++;
  }
  std::vector<uint32_t> h((size_t)words);
  CK(cudaMemcpyAsync(h.data(), d, (size_t)words * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  cudaFree(d);
  if (s2) for (int i = 0; i < c->bins2d; ++i) s2[i] = h[i];
  if (s1a) for (int i = 0; i < c->R1; ++i) s1a[i] = h[c->bins2d + i];
  if (s1b) for (int i = 0; i < c->R2; ++i) s1b[i] = h[c->bins2d + c->R1 + i];
  return 0;
}

// ------------------------------------------------------------------------------------------------ per-window passes
// Arrays of pass w for ncand windows and `parts` segments, grown after the stream has drained (a previous asynchronous
// call may still use the old ones).
static int pass_buffers(tdsfs_ctx* c, WindowPass& w, long long ncand, long long parts) {
  if (ncand > w.cap || parts > w.part_cap) CK(cudaStreamSynchronize(c->stream));
  if (ncand > w.cap) {
    free_pass_windows(w);
    CKR(dev_alloc(&w.d_wlo, ncand)); CKR(dev_alloc(&w.d_whi, ncand)); CKR(dev_alloc(&w.d_wchrom, ncand));
    CKR(dev_alloc(&w.d_count, ncand)); CKR(dev_alloc(&w.d_wstart, ncand)); CKR(dev_alloc(&w.d_wend, ncand));
    CKR(dev_alloc(&w.d_nseg, ncand + 1)); CKR(dev_alloc(&w.d_segoff, ncand + 1)); CKR(dev_alloc(&w.d_flags, ncand));
    for (int i = 0; i < w.n_i32; ++i) CKR(dev_alloc(&w.d_i32[i], ncand));
    for (int i = 0; i < w.n_f64; ++i) CKR(dev_alloc(&w.d_f64[i], ncand));
    size_t tmp = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp, w.d_nseg, w.d_segoff, (int)(ncand + 1), c->stream));
    CK(cudaMalloc(&w.d_tmp, std::max<size_t>(tmp, 16)));
    w.tmp_bytes = std::max<size_t>(tmp, 16);
    w.cap = ncand;
  }
  if (parts > w.part_cap) {
    dev_free(w.d_part);
    CK(cudaMalloc(&w.d_part, (size_t)parts * w.part_bytes));
    w.part_cap = parts;
  }
  if (!w.d_large) {
    CKR(dev_alloc(&w.d_large, 1));
    CKR(dev_alloc(&w.d_nlarge, 1));
  }
  return 0;
}

// After the rows of a host upload still in flight: window boundaries of pass w's w.ncand candidates (K2 into its own
// arrays) -> segments per window (k_div_nseg) -> the segment list (exclusive scan), on the handle's stream.
static int pass_segments(tdsfs_ctx* c, WindowPass& w, long long W, bool snp_mode) {
  cudaStream_t st = c->stream;
  for (auto& ch : c->chunks) if (ch.ev) CK(cudaStreamWaitEvent(st, ch.ev, 0));
  const long long ncand = w.ncand;
  if (ncand == 0) return 0;
  WinParams wp;
  wp.pos = c->dPos; wp.chrom_off = c->d_off; wp.cand_off = w.cand.d_off; wp.C = c->C; wp.W = W; wp.ncand = ncand;
  wp.wlo = w.d_wlo; wp.whi = w.d_whi; wp.wchrom = w.d_wchrom; wp.wstart = w.d_wstart; wp.wend = w.d_wend;
  wp.large = w.d_large; wp.nlarge = w.d_nlarge;
  wp.r_count = w.d_count; wp.r_flags = w.d_flags;  // K2 marks empty windows; the pass's finish kernel rewrites every entry
  wp.wcap = 0x7FFFFFFF;
  const int g2 = (int)((ncand + 255) / 256);
  if (snp_mode) k2_bounds_snp<<<g2, 256, 0, st>>>(wp); else k2_bounds_bp<<<g2, 256, 0, st>>>(wp);
  k_div_nseg<<<(int)((ncand + 1 + 255) / 256), 256, 0, st>>>(w.d_wlo, w.d_whi, ncand, w.d_nseg);
  size_t tmp = w.tmp_bytes;
  CK(cub::DeviceScan::ExclusiveSum(w.d_tmp, tmp, w.d_nseg, w.d_segoff, (int)(ncand + 1), st));
  c->launches += 3;
  return 0;
}

// A pass's segment kernel for the loaded rows: compile-time word counts for the genotype entry's 500 + 500 and 200 + 200
// diploid panels (BASELINE configs 5 and 4), the runtime decode for any other width and for the counts entry.
template <typename P>
static auto segment_kernel(const tdsfs_ctx* c, void (*k32)(P), void (*k14)(P), void (*k0)(P)) -> void (*)(P) {
  if (c->dG && c->W1 == 32 && c->W2 == 32) return k32;
  if (c->dG && c->W1 == 14 && c->W2 == 14) return k14;
  return k0;
}

// One per-window pass over the candidate windows of (W, mode), in the order of tdsfs_scan_*: the segment list
// (pass_segments), then launch(c, grid): the pass's params, its segment kernel on `grid` CTAs (one warp per segment of
// DIV_SEG rows; warps past the actual count return at once) and its finish kernel.  prepare (NULL: none) sets up what else
// those kernels read, before the timed range, or rejects the loaded data.  Needs loaded data only, and no host round trip
// when !fetch; when fetch, the caller fetches the results.
static int window_pass(tdsfs_ctx* c, WindowPass tdsfs_ctx::*pass, long long W, bool snp_mode, bool fetch, int64_t cap,
                       int64_t* n_windows, int (*prepare)(tdsfs_ctx*), void (*launch)(tdsfs_ctx*, unsigned)) {
  if (!c || W < 1) return fail(TDSFS_ERR_ARG, "bad argument");
  if (!c->loaded) return fail(TDSFS_ERR_STATE, "load data first");
  WindowPass& w = c->*pass;
  CK(cudaSetDevice(c->device));
  NvtxRange nvtx(w.name);
  cudaStream_t st = c->stream;
  CKR(cached_candidates(c, w.cand, W, snp_mode, st));
  const long long ncand = w.cand.off[c->C];
  if (fetch && cap < ncand) return fail(TDSFS_ERR_ARG, "result capacity %lld < %lld candidate windows", (long long)cap, ncand);
  // windows never overlap, so sum_w ceil(rows_w / SEG) <= S / SEG + ncand
  const long long max_parts = ncand + c->S / DIV_SEG + 1;
  CKR(pass_buffers(c, w, ncand, max_parts));
  if (prepare) CKR(prepare(c));
  w.ready = false;
  w.ncand = ncand;
  CKR(pass_segments(c, w, W, snp_mode));
  CK(cudaEventRecord(w.ev0, st));
  if (ncand > 0) {
    launch(c, (unsigned)((max_parts + DIV_WARPS - 1) / DIV_WARPS));
    c->launches += 2;
    CK(cudaGetLastError());
  }
  CK(cudaEventRecord(w.ev1, st));
  w.timed = true;
  w.ready = true;
  if (fetch) return 0;
  if (n_windows) *n_windows = ncand;
  return finish(c);
}

// ------------------------------------------------------------------------------------------------ diversity (Hudson FST, pi, dxy)
extern "C" int tdsfs_fetch_diversity(tdsfs_t* c, tdsfs_diversity_t* out, int64_t cap, int64_t* n_windows) {
  if (!c || !out) return fail(TDSFS_ERR_ARG, "NULL argument");
  const WindowPass& w = c->div;
  if (!w.ready) return fail(TDSFS_ERR_STATE, "no diversity results (tdsfs_diversity_bp / _snp first)");
  if (cap < w.ncand) return fail(TDSFS_ERR_ARG, "result capacity %lld < %lld candidate windows", (long long)cap, w.ncand);
  CK(cudaSetDevice(c->device));
  return fetch_columns(c, w.ncand, {{out->chrom, w.d_wchrom}, {out->start, w.d_wstart}, {out->end, w.d_wend},
                                    {out->snp_count, w.d_count}, {out->flags, w.d_flags}, {out->n_sites, w.d_i32[0]},
                                    {out->pi_p1, w.d_f64[0]}, {out->pi_p2, w.d_f64[1]}, {out->dxy, w.d_f64[2]},
                                    {out->fst, w.d_f64[3]}}, n_windows);
}

static void launch_diversity(tdsfs_ctx* c, unsigned grid) {
  const WindowPass& w = c->div;
  DivParams p;
  memset(&p, 0, sizeof p);
  fill_key_params(c, p.k);
  p.seg = w.segs(); p.part = (DivPart*)w.d_part; p.snp_count = w.d_count; p.flags = w.d_flags; p.n_sites = w.d_i32[0];
  p.pi1 = w.d_f64[0]; p.pi2 = w.d_f64[1]; p.dxy = w.d_f64[2]; p.fst = w.d_f64[3];
  const auto kern = segment_kernel(c, k_diversity<32, 32>, k_diversity<14, 14>, k_diversity<0, 0>);
  kern<<<grid, DIV_WARPS * 32, 0, c->stream>>>(p);
  k_div_finish<<<(int)((w.ncand + 255) / 256), 256, 0, c->stream>>>(p);
}

// Per-window Hudson FST, pi and dxy: k_diversity -> k_div_finish.
static int diversity(tdsfs_ctx* c, long long W, bool snp_mode, tdsfs_diversity_t* out, int64_t cap, int64_t* n_windows) {
  CKR(window_pass(c, &tdsfs_ctx::div, W, snp_mode, out != nullptr, cap, n_windows, nullptr, launch_diversity));
  return out ? tdsfs_fetch_diversity(c, out, cap, n_windows) : 0;
}

extern "C" int tdsfs_diversity_bp(tdsfs_t* c, int64_t W, tdsfs_diversity_t* out, int64_t cap, int64_t* n_windows) {
  return diversity(c, W, false, out, cap, n_windows);
}
extern "C" int tdsfs_diversity_snp(tdsfs_t* c, int64_t N, tdsfs_diversity_t* out, int64_t cap, int64_t* n_windows) {
  return diversity(c, N, true, out, cap, n_windows);
}

// ------------------------------------------------------------------------------------------------ neutrality (theta_W, Tajima's D)
extern "C" int tdsfs_fetch_neutrality(tdsfs_t* c, tdsfs_neutrality_t* out, int64_t cap, int64_t* n_windows) {
  if (!c || !out) return fail(TDSFS_ERR_ARG, "NULL argument");
  const WindowPass& w = c->neut;
  if (!w.ready) return fail(TDSFS_ERR_STATE, "no neutrality results (tdsfs_neutrality_bp / _snp first)");
  if (cap < w.ncand) return fail(TDSFS_ERR_ARG, "result capacity %lld < %lld candidate windows", (long long)cap, w.ncand);
  CK(cudaSetDevice(c->device));
  return fetch_columns(c, w.ncand, {{out->chrom, w.d_wchrom}, {out->start, w.d_wstart}, {out->end, w.d_wend},
                                    {out->snp_count, w.d_count}, {out->flags, w.d_flags}, {out->n_seg_p1, w.d_i32[0]},
                                    {out->n_seg_p2, w.d_i32[1]}, {out->n_max_p1, w.d_i32[2]}, {out->n_max_p2, w.d_i32[3]},
                                    {out->theta_pi_p1, w.d_f64[0]}, {out->theta_pi_p2, w.d_f64[1]},
                                    {out->theta_w_p1, w.d_f64[2]}, {out->theta_w_p2, w.d_f64[3]},
                                    {out->tajima_d_p1, w.d_f64[4]}, {out->tajima_d_p2, w.d_f64[5]}}, n_windows);
}

// a1(n) and a2(n) for every n a loaded row can reach, summed in ascending k; built again only when a load reaches a
// larger n (the entries of a longer table are the same numbers)
static int neut_table(tdsfs_ctx* c) {
  if (c->n_allele_max <= c->neut_tab_n) return 0;
  const long long m = c->n_allele_max + 1;
  std::vector<double> t((size_t)(2 * m), 0.0);
  for (long long n = 2; n < m; ++n) {
    const double k = (double)(n - 1);
    t[n] = t[n - 1] + 1.0 / k;
    t[m + n] = t[m + n - 1] + 1.0 / (k * k);
  }
  CK(cudaStreamSynchronize(c->stream));  // a previous asynchronous call may still read the old table
  c->neut_tab_n = -1;
  dev_free(c->d_neut_tab);
  CKR(dev_alloc(&c->d_neut_tab, 2 * m));
  CK(cudaMemcpyAsync(c->d_neut_tab, t.data(), (size_t)(2 * m) * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  c->neut_tab_n = m - 1;
  return 0;
}

static void launch_neutrality(tdsfs_ctx* c, unsigned grid) {
  const WindowPass& w = c->neut;
  NeutParams p;
  memset(&p, 0, sizeof p);
  fill_key_params(c, p.k);
  p.seg = w.segs(); p.part = (NeutPart*)w.d_part; p.snp_count = w.d_count; p.flags = w.d_flags;
  p.a1 = c->d_neut_tab; p.a2 = c->d_neut_tab + c->neut_tab_n + 1;
  p.S1 = w.d_i32[0]; p.S2 = w.d_i32[1]; p.nmax1 = w.d_i32[2]; p.nmax2 = w.d_i32[3];
  p.theta_pi1 = w.d_f64[0]; p.theta_pi2 = w.d_f64[1]; p.theta_w1 = w.d_f64[2]; p.theta_w2 = w.d_f64[3];
  p.tajd1 = w.d_f64[4]; p.tajd2 = w.d_f64[5];
  const auto kern = segment_kernel(c, k_neutrality<32, 32>, k_neutrality<14, 14>, k_neutrality<0, 0>);
  kern<<<grid, DIV_WARPS * 32, 0, c->stream>>>(p);
  k_neut_finish<<<(int)((w.ncand + 255) / 256), 256, 0, c->stream>>>(p);
}

// Per-window, per-population Watterson's theta and Tajima's D: k_neutrality -> k_neut_finish.  The first call after a load
// that needs a larger a1 / a2 table waits for the stream once.
static int neutrality(tdsfs_ctx* c, long long W, bool snp_mode, tdsfs_neutrality_t* out, int64_t cap, int64_t* n_windows) {
  CKR(window_pass(c, &tdsfs_ctx::neut, W, snp_mode, out != nullptr, cap, n_windows, neut_table, launch_neutrality));
  return out ? tdsfs_fetch_neutrality(c, out, cap, n_windows) : 0;
}

extern "C" int tdsfs_neutrality_bp(tdsfs_t* c, int64_t W, tdsfs_neutrality_t* out, int64_t cap, int64_t* n_windows) {
  return neutrality(c, W, false, out, cap, n_windows);
}
extern "C" int tdsfs_neutrality_snp(tdsfs_t* c, int64_t N, tdsfs_neutrality_t* out, int64_t cap, int64_t* n_windows) {
  return neutrality(c, N, true, out, cap, n_windows);
}

// ------------------------------------------------------------------------------------------------ Weir and Cockerham's FST
extern "C" int tdsfs_fetch_wcfst(tdsfs_t* c, tdsfs_wcfst_t* out, int64_t cap, int64_t* n_windows) {
  if (!c || !out) return fail(TDSFS_ERR_ARG, "NULL argument");
  const WindowPass& w = c->wc;
  if (!w.ready) return fail(TDSFS_ERR_STATE, "no Weir and Cockerham FST results (tdsfs_wcfst_bp / _snp first)");
  if (cap < w.ncand) return fail(TDSFS_ERR_ARG, "result capacity %lld < %lld candidate windows", (long long)cap, w.ncand);
  CK(cudaSetDevice(c->device));
  return fetch_columns(c, w.ncand, {{out->chrom, w.d_wchrom}, {out->start, w.d_wstart}, {out->end, w.d_wend},
                                    {out->snp_count, w.d_count}, {out->flags, w.d_flags}, {out->n_sites, w.d_i32[0]},
                                    {out->a, w.d_f64[0]}, {out->b, w.d_f64[1]}, {out->c, w.d_f64[2]},
                                    {out->fst, w.d_f64[3]}}, n_windows);
}

// The pass reads heterozygote counts, which only the 2-bit calls hold, and its int64 terms are exact up to WC_MAX_SAMPLES
// samples per population.
static int wc_check(tdsfs_ctx* c) {
  if (!c->genotypes)
    return fail(TDSFS_ERR_STATE, "Weir and Cockerham FST needs genotype calls (tdsfs_load_genotypes): the counts entry has no heterozygote counts");
  if (c->ns1 > WC_MAX_SAMPLES || c->ns2 > WC_MAX_SAMPLES)
    return fail(TDSFS_ERR_ARG, "Weir and Cockerham FST takes at most %d samples per population (%d + %d loaded): its int64 terms would overflow",
                WC_MAX_SAMPLES, c->ns1, c->ns2);
  return 0;
}

static void launch_wcfst(tdsfs_ctx* c, unsigned grid) {
  const WindowPass& w = c->wc;
  WcParams p;
  memset(&p, 0, sizeof p);
  fill_key_params(c, p.k);
  p.seg = w.segs(); p.part = (WcPart*)w.d_part; p.snp_count = w.d_count; p.flags = w.d_flags; p.n_sites = w.d_i32[0];
  p.a = w.d_f64[0]; p.b = w.d_f64[1]; p.c = w.d_f64[2]; p.fst = w.d_f64[3];
  const auto kern = segment_kernel(c, k_wcfst<32, 32>, k_wcfst<14, 14>, k_wcfst<0, 0>);
  kern<<<grid, DIV_WARPS * 32, 0, c->stream>>>(p);
  k_wc_finish<<<(int)((w.ncand + 255) / 256), 256, 0, c->stream>>>(p);
}

// Per-window Weir and Cockerham FST from the genotype calls: k_wcfst -> k_wc_finish.
static int wcfst(tdsfs_ctx* c, long long W, bool snp_mode, tdsfs_wcfst_t* out, int64_t cap, int64_t* n_windows) {
  CKR(window_pass(c, &tdsfs_ctx::wc, W, snp_mode, out != nullptr, cap, n_windows, wc_check, launch_wcfst));
  return out ? tdsfs_fetch_wcfst(c, out, cap, n_windows) : 0;
}

extern "C" int tdsfs_wcfst_bp(tdsfs_t* c, int64_t W, tdsfs_wcfst_t* out, int64_t cap, int64_t* n_windows) {
  return wcfst(c, W, false, out, cap, n_windows);
}
extern "C" int tdsfs_wcfst_snp(tdsfs_t* c, int64_t N, tdsfs_wcfst_t* out, int64_t cap, int64_t* n_windows) {
  return wcfst(c, N, true, out, cap, n_windows);
}

// ------------------------------------------------------------------------------------------------ LD pruning
// k_ld_pairs (the pair bits of every row) -> k_ld_resolve (the greedy decision per chromosome), then the keep bytes and the
// kept count to the host.  Synchronous.
extern "C" int tdsfs_ld_prune(tdsfs_t* c, int32_t size, int32_t step, double threshold, uint8_t* keep, int64_t* n_kept) {
  if (!c || !keep) return fail(TDSFS_ERR_ARG, "ctx / keep is NULL");
  if (size < 2 || size > LD_MAX_SIZE || step < 1 || !std::isfinite(threshold) || threshold < 0.0 || threshold > 1.0)
    return fail(TDSFS_ERR_ARG, "LD pruning takes 2 <= size <= %d, step >= 1 and a threshold in [0, 1] (got %d, %d, %g)",
                LD_MAX_SIZE, size, step, threshold);
  if (!c->loaded) return fail(TDSFS_ERR_STATE, "load data first");
  if (!c->genotypes)
    return fail(TDSFS_ERR_STATE, "LD pruning needs genotype calls (tdsfs_load_genotypes): the counts entry has no calls");
  CK(cudaSetDevice(c->device));
  NvtxRange nvtx("tdsfs:LD pruning");
  cudaStream_t st = c->stream;
  for (auto& ch : c->chunks) if (ch.ev) CK(cudaStreamWaitEvent(st, ch.ev, 0));
  const long long S = c->S;
  const int mw = (size - 1 + 31) / 32;
  // the previous call ended with a synchronise: nothing still reads the old buffers
  if (S * mw > c->ld_mask_cap) {
    dev_free(c->d_ld_mask);
    c->ld_mask_cap = 0;
    CKR(dev_alloc(&c->d_ld_mask, S * mw));
    c->ld_mask_cap = S * mw;
  }
  if (S > c->ld_keep_cap) {
    dev_free(c->d_ld_keep);
    c->ld_keep_cap = 0;
    CKR(dev_alloc(&c->d_ld_keep, S));
    c->ld_keep_cap = S;
  }
  LdParams p;
  memset(&p, 0, sizeof p);
  p.G = c->dG; p.S = S; p.W1 = c->W1; p.W2 = c->W2; p.ns1 = c->ns1; p.ns2 = c->ns2;
  p.chrom_off = c->d_off; p.C = c->C;
  p.size = size; p.step = step; p.mw = mw; p.thr = threshold;
  p.mask = c->d_ld_mask; p.keep = c->d_ld_keep; p.n_kept = c->d_ld_n;
  CK(cudaMemsetAsync(c->d_ld_n, 0, sizeof(unsigned long long), st));
  CK(cudaEventRecord(c->ev_ld[0], st));
  if (S > 0) {
    const auto kern = segment_kernel(c, k_ld_pairs<32, 32>, k_ld_pairs<14, 14>, k_ld_pairs<0, 0>);
    kern<<<(unsigned)((S + BLK - 1) / BLK), LD_WARPS * 32, 0, st>>>(p);
    CK(cudaEventRecord(c->ev_ld[1], st));
    k_ld_resolve<<<c->C, 32, 0, st>>>(p);
    c->launches += 2;
    CK(cudaGetLastError());
  } else {
    CK(cudaEventRecord(c->ev_ld[1], st));
  }
  CK(cudaEventRecord(c->ev_ld[2], st));
  c->ld_timed = true;
  unsigned long long nk = 0;
  if (S > 0) CK(cudaMemcpyAsync(keep, c->d_ld_keep, (size_t)S, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&nk, c->d_ld_n, sizeof nk, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (n_kept) *n_kept = (int64_t)nk;
  return 0;
}

// ------------------------------------------------------------------------------------------------ explicit likelihood
extern "C" int tdsfs_likelihood(tdsfs_t* c, const int64_t* x, const double* b, int64_t n, double B, double* T, int32_t* flag) {
  if (!c || !T || !flag || n < 0 || (n > 0 && (!x || !b))) return fail(TDSFS_ERR_ARG, "bad argument");
  CK(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  long long* dx = nullptr;
  double *db = nullptr, *dout = nullptr;
  int* dflag = nullptr;
  CKR(dev_alloc(&dx, n)); CKR(dev_alloc(&db, n)); CKR(dev_alloc(&dout, 1)); CKR(dev_alloc(&dflag, 1));
  if (n) {
    CK(cudaMemcpyAsync(dx, x, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(db, b, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  }
  k_likelihood<<<1, 256, 0, st>>>(dx, db, n, B, dout, dflag);
  c->launches++;
  CK(cudaGetLastError());
  int hf = 0;
  CK(cudaMemcpyAsync(T, dout, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&hf, dflag, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  *flag = hf;
  cudaFree(dx); cudaFree(db); cudaFree(dout); cudaFree(dflag);
  return 0;
}

extern "C" int tdsfs_poisson_score(tdsfs_t* c, const int64_t* x, const double* mu, int64_t n, double* score) {
  if (!c || !score || n < 0 || (n > 0 && (!x || !mu))) return fail(TDSFS_ERR_ARG, "bad argument");
  CK(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  long long* dx = nullptr;
  double *dm = nullptr, *dout = nullptr;
  CKR(dev_alloc(&dx, n)); CKR(dev_alloc(&dm, n)); CKR(dev_alloc(&dout, 1));
  if (n) {
    CK(cudaMemcpyAsync(dx, x, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(dm, mu, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  }
  k_poisson<<<1, 256, 0, st>>>(dx, dm, n, dout);
  c->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(score, dout, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  cudaFree(dx); cudaFree(dm); cudaFree(dout);
  return 0;
}

// ------------------------------------------------------------------------------------------------ synthetic + instrumentation
extern "C" int tdsfs_synth_genotypes(tdsfs_t* c, void* G_dev, int64_t S, int64_t snp0, int32_t words1, int32_t words2,
                                     int32_t ns1, int32_t ns2, uint64_t seed, double missing_rate, double fst) {
  if (!c || !G_dev || S < 0) return fail(TDSFS_ERR_ARG, "bad argument");
  if (!is_device_ptr(G_dev)) return fail(TDSFS_ERR_ARG, "G_dev must be device memory");
  CK(cudaSetDevice(c->device));
  // every word of every 32-SNP block, padding rows included: in the block-transposed layout the words of the second population of
  // a partial last block lie beyond S * RW (found by the bench line's cross-N checksums: they were left uninitialised)
  const long long total = (S + BLK - 1) / BLK * BLK * (long long)(words1 + words2);
  const uint32_t thr = (uint32_t)(missing_rate * 65536.0);
  const long long blocks = (total + 255) / 256;
  if (blocks > 0x7FFFFFFFLL) return fail(TDSFS_ERR_ARG, "matrix too large for one launch");
  if (blocks) {
    k_synth<<<(unsigned)blocks, 256, 0, c->stream>>>((uint32_t*)G_dev, S, snp0, words1, words2, ns1, ns2, seed, thr, fst);
    c->launches++;
  }
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int tdsfs_timings(tdsfs_t* c, float* ms, int32_t n) {
  if (!c || !ms) return fail(TDSFS_ERR_ARG, "NULL argument");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  for (int i = 0; i < 14; ++i) c->ms[i] = 0.f;
  if (c->keys_ready) cudaEventElapsedTime(&c->ms[0], c->ev[EV_BG0], c->ev[EV_K1]);
  if (c->fin_timed) cudaEventElapsedTime(&c->ms[1], c->ev[EV_FIN0], c->ev[EV_FIN1]);
  if (c->results_ready) {
    if (c->planned_last) cudaEventElapsedTime(&c->ms[2], c->ev_plan0, c->ev_plan);  // K2 ran on the side stream
    else cudaEventElapsedTime(&c->ms[2], c->ev[EV_SC0], c->ev[EV_K2]);
    cudaEventElapsedTime(&c->ms[3], c->ev[EV_K2], c->ev[EV_K3S]);
    cudaEventElapsedTime(&c->ms[4], c->ev[EV_K3S], c->ev[EV_K3L]);
    cudaEventElapsedTime(&c->ms[6], c->ev[EV_SC0], c->ev[EV_K3L]);
    if (c->keys_ready) cudaEventElapsedTime(&c->ms[7], c->ev[EV_BG0], c->ev[EV_K3L]);
  }
  c->ms[5] = c->ms[0];
  if (c->x_timed) cudaEventElapsedTime(&c->ms[8], c->ev[EV_X0], c->ev[EV_X1]);
  if (c->div.timed) cudaEventElapsedTime(&c->ms[9], c->div.ev0, c->div.ev1);
  if (c->neut.timed) cudaEventElapsedTime(&c->ms[10], c->neut.ev0, c->neut.ev1);
  if (c->wc.timed) cudaEventElapsedTime(&c->ms[11], c->wc.ev0, c->wc.ev1);
  if (c->ld_timed) {
    cudaEventElapsedTime(&c->ms[12], c->ev_ld[0], c->ev_ld[1]);
    cudaEventElapsedTime(&c->ms[13], c->ev_ld[1], c->ev_ld[2]);
  }
  cudaGetLastError();
  for (int i = 0; i < n && i < 14; ++i) ms[i] = c->ms[i];
  return 0;
}

extern "C" int64_t tdsfs_launch_count(tdsfs_t* c) { return c ? c->launches : 0; }

extern "C" int tdsfs_tail_stamps(tdsfs_t* c, uint64_t* out8) {
  if (!c || !out8) return fail(TDSFS_ERR_ARG, "ctx or out is NULL");
  if (!c->d_stamps) return fail(TDSFS_ERR_STATE, "tail stamps are off (create the handle with TDSFS_TAIL_STAMPS=1 set)");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaMemcpy(out8, c->d_stamps, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int tdsfs_scan_info(tdsfs_t* c, int32_t* fused, int32_t* record_bytes) {
  if (!c) return fail(TDSFS_ERR_ARG, "ctx is NULL");
  if (fused) *fused = c->last_fused ? 1 : 0;
  if (record_bytes) *record_bytes = c->fmt.narrow ? 4 : 8;
  return 0;
}
