// apgk.cu -- context, host orchestration and the C ABI (include/apgk.h) of libapgk.so.
//
// Pipeline of apgk_finish (one GPU, see DESIGN.md):
//   level 0   k_hist_reads -> column scan -> k_scatter_reads   reads  -> A (full keys, bucketed by D0 bits)
//   level 1   k_hist_keys  -> column scan -> k_scatter_keys    A      -> B (remainders or full keys, D1 bits)
//   local     k_local (+ k_big for oversize buckets)           B      -> temp records in A/B + spectrum
//   table     scan of per-bucket record counts -> k_compact    temp   -> sorted (k-mer, count) table + index
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <map>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/apgk.h"
#include "gfreq.cuh"

using namespace apgk;

namespace {

enum Stage { ST_HIST0, ST_SCAN0, ST_SCATTER0, ST_HIST1, ST_SCAN1, ST_SCATTER1, ST_LOCAL, ST_BIG, ST_TABLE, ST_SPECTRUM,
             ST_OWNER, ST_TOTAL, ST_PLAN, ST_REDUCE };
// owner = the gather of the sharded form; plan = its all-gather + splitters (includes waiting for slower ranks);
// reduce = the spectrum all-reduce (ditto)
const char* kStageNames[APGK_N_STAGES] = {"hist0", "scan0", "scatter0", "hist1", "scan1", "scatter1",
                                          "local", "big", "table", "spectrum", "owner", "total", "plan", "reduce"};

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  // NOTE: cudaMemset / cudaMemcpy(D2D) on the legacy stream do not order with the context's
  // non-blocking stream, so zeroing synchronises the device before returning.
  cudaError_t ensure(size_t bytes, bool zero_new = false) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + (bytes >> 5) + 4096;  // a little slack so small growth does not realloc
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) { want = bytes; e = cudaMalloc(&p, want); }
    if (e != cudaSuccess) { p = nullptr; return e; }
    cap = want;
    if (zero_new) {
      e = cudaMemset(p, 0, cap);
      if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename T> T* as() const { return (T*)p; }
};

// host-side description of a partition level, mirrored on the device in ctx->plan
struct HostPlan {
  std::vector<uint32_t> seg_tile0, seg_chunk0;
  std::vector<uint64_t> seg_start;
  LevelPlan lp{};
};

}  // namespace

struct apgk_group;
struct apgk_ctx {
  apgk_config cfg{};
  apgk_group* group = nullptr;       // the group this context is a member of (include/apgk.h "a GROUP of ranks")
  uint64_t gen = 0;                  // bumped by every call that changes the read store or the table
  int W = 1;
  int device = 0;
  int n_sm = 148;
  cudaStream_t stream = nullptr;
  std::string err;
  // ---- read store
  DevBuf bases, starts, staging, off_dev;
  uint64_t total_bases = 0, n_reads = 0;
  uint64_t n_windows = 0;            // exact k-mer instances of the store: sum over reads of max(0, L - K + 1)
  uint64_t n_windows_run = 0;        // instances the current step's level-0 histogram must find (store, or a key array)
  // ---- streamed ingest (APGK_ASYNC_INGEST): copies in flight on copy_stream, one event per slice
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_main = nullptr;
  std::vector<cudaEvent_t> slice_ev;
  std::vector<uint64_t> slice_end;   // bases resident once slice i has landed
  size_t n_slices = 0;               // pending slices (0 = nothing in flight)
  // ---- pipeline buffers
  DevBuf tot0_dev, res;              // level-0 bucket totals; the step's result block (RES_*)
  unsigned long long* res_host = nullptr;   // pinned mirror of `res`
  HostPlan hp0;                      // level-0 plan: a function of the input size, kept from step to step
  uint64_t hp0_elems = ~0ull; uint32_t hp0_tile = 0;
  std::map<std::pair<const void*, size_t>, int> kattr;   // (kernel, dynamic smem) -> occupancy, attribute set
  double table_scale = 1.0;          // rounds: instances of the whole run over instances counted so far (table growth hint)
  bool table_pending = false;        // single-round step: the table's size is read at the final synchronisation
  void* tmp_keys_last = nullptr;     // where the last count_buckets left its per-bucket records
  DevBuf A, B, T, chunksum, chunksum0, plan0, out_off_local, segtot, bstart32, bofs, plan, bstart64, nd, out_off, blocksum, big_list, stats,
      scratch, stacks, spec_dense, spec_ovf, misc, deferred;
  // ---- results
  DevBuf out_keys, out_cnt;
  bool finished = false, have_table = false;
  bool table_from_reads = false;   // the table counts exactly the windows of this context's read store
  // ---- occurrence records (apgk_build_occurrences): run offsets + (position << 1 | rc) per instance, in A
  DevBuf occ, occ_pos, occ_off, occ_cnt, occ_bstart, occ_bcur, rank_cnt, rank_dir, empty_dev, occ_tmp;
  bool have_occ = false;
  uint64_t n_occ = 0, n_big_runs = 0;
  float occ_ms[5]{};
  float freq_ms[3]{};              // last bulk read_freqs: {memset + scan, sweep, placement}
  cudaEvent_t occ_ev[6]{};
  std::vector<uint64_t> empty_nb;  // per read without bases: number of reads WITH bases before it
  uint64_t n_instances = 0, n_distinct = 0;
  KeyGeom geom{};
  uint32_t nb1 = 0;          // number of level-1 buckets
  uint32_t elem_bytes = 0;   // level-1 element size
  uint64_t n_big = 0;
  uint32_t n_deferred = 0, local_max = 0, n_rounds = 0;
  std::vector<uint64_t> spec_host, sparse_f, sparse_n;
  bool spec_loaded = false;
  // ---- partition-only state (sharded counting: apgk_partition -> exchange -> apgk_count_pieces)
  int force_d0_lo = -1, force_d0_hi = -1;   // apgk_partition_range: the one k-mer-space round to partition
  std::vector<uint64_t> tot0_host;          // level-0 bucket totals of the last run over the read store
  uint64_t last_cap_keys = 0;               // k-mer instances one round may hold (memory budget of the last run)
  bool part_ready = false;
  uint64_t part_n = 0;       // elements in B, grouped by the nb1 buckets (sizes in segtot)
  DevBuf piece_off, piece_tmp, piece_ptrs, C2, sub_sizes, TK;
  uint64_t budget_bytes = 0, budget_for = 0;   // temp-buffer budget of the sharded form, and the store size it was asked for
  void* count_src = nullptr;
  uint32_t bucket_lo = 0, bucket_hi = 0;  // shard's bucket range for count_buckets (0,0 = all)  // elements count_buckets reads (B, or C2 on the peer-memory path)
  // ---- owner partition state
  uint32_t owner_ranks = 0;
  uint32_t owner_tiles = 0;
  std::vector<uint64_t> owner_counts;
  HostPlan owner_plan;
  DevBuf owner_plan_dev;
  // ---- instrumentation: one (start, end) event pair per stage interval of the current step, taken from a
  // pool and read back at the step's final synchronisation (a stage may run many times per step)
  struct StageIv { int stage; cudaEvent_t e0, e1; bool ended; };
  std::vector<StageIv> ivs;
  size_t n_ivs = 0;
  int open_iv[APGK_N_STAGES]{};
  float stage_ms[APGK_N_STAGES]{};
  uint64_t launches = 0;
};

namespace {

#define CU(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e__ = (call);                                                                            \
    if (e__ != cudaSuccess) {                                                                            \
      char b__[512];                                                                                     \
      snprintf(b__, sizeof b__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
      c->err = b__;                                                                                      \
      return (e__ == cudaErrorMemoryAllocation) ? APGK_E_NOMEM : APGK_E_CUDA;                            \
    }                                                                                                    \
  } while (0)

#define FAIL(code, ...)                        \
  do {                                         \
    char b__[512];                             \
    snprintf(b__, sizeof b__, __VA_ARGS__);    \
    c->err = b__;                              \
    return (code);                             \
  } while (0)

static const bool kSyncDebug = getenv("APGK_SYNC_DEBUG") != nullptr;  // sync after every launch to localise faults
#define LAUNCHED() do { c->launches++; CU(cudaGetLastError()); if (kSyncDebug) CU(cudaStreamSynchronize(c->stream)); } while (0)

// Stage intervals are recorded without ever waiting on the device mid-step; stages_collect() folds them into
// stage_ms once the step's stream has been synchronised.
static const bool kTrace = getenv("APGK_TRACE") != nullptr;  // host wall clock at every stage boundary, to stderr
static double trace_now() {
  timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
void stages_reset(apgk_ctx* c) {
  c->n_ivs = 0;
  for (int s = 0; s < APGK_N_STAGES; s++) { c->stage_ms[s] = 0; c->open_iv[s] = -1; }
}
void stage_begin(apgk_ctx* c, int s) {
  if (c->n_ivs == c->ivs.size()) {
    apgk_ctx::StageIv iv{s, nullptr, nullptr, false};
    if (cudaEventCreate(&iv.e0) != cudaSuccess || cudaEventCreate(&iv.e1) != cudaSuccess) return;
    c->ivs.push_back(iv);
  }
  apgk_ctx::StageIv& iv = c->ivs[c->n_ivs];
  iv.stage = s; iv.ended = false;
  c->open_iv[s] = (int)c->n_ivs++;
  if (kTrace) fprintf(stderr, "[apgk %.2f] begin %s\n", trace_now(), kStageNames[s]);
  cudaEventRecord(iv.e0, c->stream);
}
void stage_end(apgk_ctx* c, int s) {
  const int i = c->open_iv[s];
  if (i < 0) return;
  cudaEventRecord(c->ivs[i].e1, c->stream);
  c->ivs[i].ended = true;
  c->open_iv[s] = -1;
  if (kTrace) fprintf(stderr, "[apgk %.2f] end   %s\n", trace_now(), kStageNames[s]);
}
// after the stream has been synchronised
void stages_collect(apgk_ctx* c) {
  for (size_t i = 0; i < c->n_ivs; i++) {
    float ms = 0;
    if (c->ivs[i].ended && cudaEventElapsedTime(&ms, c->ivs[i].e0, c->ivs[i].e1) == cudaSuccess) c->stage_ms[c->ivs[i].stage] += ms;
  }
  c->n_ivs = 0;
}

int words_for(int K) { return (2 * K + 63) / 64; }

// tile geometry per key width
template <int W> struct Geo;
// NT0: threads of a level-0 CTA (16 windows each); NT1 / TILE1: threads and keys of a key-array tile
// (TILE1 == NT1 * TileItems<Key<W>>::N, the keys live in registers during ranking)
#ifndef APGK_NT
#define APGK_NT 1024
#endif
// NTS / NPOS: threads and window starts per thread of the level-0 SCATTER (NTS * NPOS == NT0 * 16: same tiles as the histogram)
template <> struct Geo<1> { static constexpr int NTS = APGK_NT; static constexpr int NPOS = 16; static constexpr int NT0 = APGK_NT; static constexpr int NT1 = APGK_NT; static constexpr uint32_t TILE1 = APGK_NT * 16; static constexpr int LM_KEY = 4096; };
template <> struct Geo<2> { static constexpr int NTS = 1024; static constexpr int NPOS = 8; static constexpr int NT0 = 512; static constexpr int NT1 = 512; static constexpr uint32_t TILE1 = 512 * 8;  static constexpr int LM_KEY = 2048; };
template <> struct Geo<3> { static constexpr int NTS = 1024; static constexpr int NPOS = 4; static constexpr int NT0 = 256; static constexpr int NT1 = 512; static constexpr uint32_t TILE1 = 512 * 5;  static constexpr int LM_KEY = 2048; };
constexpr int LM_U32 = 5120;
constexpr int LM_KEY4 = 3072;   // k_local4 (full-key elements): 12 bytes per slot, three CTAs per SM
// k_local4 is used for one-word keys only (K = 27..32).  For multi-word k-mers at high coverage its
// monotone rows overflow all the time: the sequencing-error variants of one genomic window share their
// leading ~26+ bases, i.e. they are ~10 distinct keys that belong in the SAME row (K=96, 24 M x 250 bp:
// 2.4 row overflows per bucket, 9 s) -- those keep the k_local2 / k_local / k_big path.  APGK_LOCAL4=all
// forces it everywhere (tests), APGK_NO_LOCAL4 switches it off.
static bool use_local4(int W) {
  static const bool off = getenv("APGK_NO_LOCAL4") != nullptr;
  static const bool all = getenv("APGK_LOCAL4") != nullptr && !strcmp(getenv("APGK_LOCAL4"), "all");
  return !off && (W == 1 || all);
}
constexpr int L3_NT = 512;
constexpr int COL_NT = 1024;

void build_plan(HostPlan& hp, const std::vector<uint64_t>& seg_sizes, uint32_t tile_elems, int bins) {
  const int S = (int)seg_sizes.size();
  hp.seg_tile0.assign(S + 1, 0); hp.seg_chunk0.assign(S + 1, 0); hp.seg_start.assign(S + 1, 0);
  uint64_t max_tiles = 1;
  for (int s = 0; s < S; s++) {
    uint64_t t = (seg_sizes[s] + tile_elems - 1) / tile_elems;
    hp.seg_tile0[s + 1] = hp.seg_tile0[s] + (uint32_t)t;
    hp.seg_start[s + 1] = hp.seg_start[s] + seg_sizes[s];
    max_tiles = std::max(max_tiles, t);
  }
  // a scatter CTA walks one chunk of tiles; ~4+ chunks per segment keep the CTAs balanced
  int ct = (int)((max_tiles + 3) / 4);
  ct = std::max(8, std::min(ct, 128));
  if (const char* e = getenv("APGK_CT")) { if (atoi(e) > 0) ct = atoi(e); }  // tuning knob
  for (int s = 0; s < S; s++) {
    uint32_t t = hp.seg_tile0[s + 1] - hp.seg_tile0[s];
    hp.seg_chunk0[s + 1] = hp.seg_chunk0[s] + (t + ct - 1) / ct;
  }
  hp.lp.bins = bins; hp.lp.n_segments = S; hp.lp.chunk_tiles = ct;
  hp.lp.n_tiles = hp.seg_tile0[S]; hp.lp.n_chunks = hp.seg_chunk0[S]; hp.lp.tile_elems = tile_elems;
}

// per-chunk digit counts (chunksum, written by the hist kernels) -> per-chunk exclusive prefixes,
// bucket totals (segtot), bucket starts inside their segment (bstart32), optional absolute bucket offsets
int column_scan(apgk_ctx* c, const HostPlan& hp, int fold, unsigned long long* bofs_out) {
  const LevelPlan& lp = hp.lp;
  if (lp.n_chunks == 0) return APGK_OK;
  CU(c->segtot.ensure((size_t)lp.n_segments * lp.bins * 8));
  CU(c->bstart32.ensure((size_t)lp.n_segments * lp.bins * 4));
  k_segscan<COL_NT><<<lp.n_segments, COL_NT, 0, c->stream>>>(lp, c->chunksum.as<uint32_t>(),
                                                            c->segtot.as<unsigned long long>(),
                                                            c->bstart32.as<uint32_t>(), bofs_out, fold);
  LAUNCHED();
  return APGK_OK;
}

template <typename K>
int set_smem(apgk_ctx* c, K kernel, size_t bytes) {
  if (bytes > 48 * 1024) CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return APGK_OK;
}

ReadStore read_store(const apgk_ctx* c) {
  ReadStore rs;
  rs.bases32 = c->bases.as<uint32_t>();
  rs.starts32 = c->starts.as<uint32_t>();
  rs.total_bases = c->total_bases;
  rs.K = c->cfg.K;
  return rs;
}

// streamed ingest: make the context's stream wait for every copy still in flight
int wait_ingest(apgk_ctx* c) {
  if (c->n_slices) {
    CU(cudaStreamWaitEvent(c->stream, c->slice_ev[c->n_slices - 1], 0));
    c->n_slices = 0;
  }
  return APGK_OK;
}

int choose_prefix_bits(const apgk_ctx* c, uint64_t upper, int local_max, bool l3) {
  if (c->cfg.prefix_bits > 0) return std::max(2, std::min(24, (int)c->cfg.prefix_bits));
  const char* env = getenv("APGK_PREFIX_BITS");
  if (env && atoi(env) > 0) return std::max(2, std::min(24, atoi(env)));
  // k_local3 (32-bit remainders) likes the average bucket near its table's key capacity: duplicates share a
  // slot and oversize ranges are split (measured best on B200: P=20 for 4.56 G k-mers, profiles/r01_sweeps.txt).  The general kernels cannot
  // split, and the densest prefixes (AAAA...) hold ~2x the average bucket, so they aim at capacity / 2.2.
  double target = l3 ? local_max * 1.0 : local_max / 2.2;
  int P = 2;
  while (P < 24 && (double)upper / (double)(1ull << P) > target) P++;
  return P;
}

// geometry for this run
void make_geom(apgk_ctx* c, int P) {
  KeyGeom& g = c->geom;
  g.K = c->cfg.K; g.W = c->W;
  g.TB = std::max(2 * g.K, P);
  g.pad = g.TB - 2 * g.K;
  g.D0 = (P + 1) / 2;
  if (const char* e = getenv("APGK_D0")) { if (atoi(e) >= 1 && atoi(e) < P && atoi(e) <= 12 && P - atoi(e) <= 12) g.D0 = atoi(e); }  // tuning knob
  g.D1 = P - g.D0;
  g.REM = g.TB - P;
  g.topbits = 2 * g.K - 64 * (g.W - 1);
}

int ensure_store(apgk_ctx* c, uint64_t bases_needed) {
  // bases: 2 bits each + 64 bytes of zero padding; starts: 1 bit each + padding.  Grow by copy.
  const size_t bbytes = ((bases_needed + 31) / 32) * 8 + 256;
  const size_t sbytes = ((bases_needed + 31) / 32) * 4 + 256;
  if (bbytes > c->bases.cap) {
    DevBuf nb, ns;
    size_t grow = std::max(bbytes, c->bases.cap * 2);
    CU(cudaStreamSynchronize(c->stream));
    cudaError_t e = nb.ensure(grow, true);
    if (e == cudaSuccess) e = ns.ensure(grow / 2 + 256, true);
    if (e == cudaSuccess && c->total_bases) {
      e = cudaMemcpyAsync(nb.p, c->bases.p, ((c->total_bases + 31) / 32) * 8 + 8, cudaMemcpyDeviceToDevice, c->stream);
      if (e == cudaSuccess) e = cudaMemcpyAsync(ns.p, c->starts.p, ((c->total_bases + 31) / 32) * 4 + 8, cudaMemcpyDeviceToDevice, c->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    }
    if (e != cudaSuccess) { nb.release(); ns.release(); }   // the old store stays in place
    CU(e);
    c->bases.release(); c->starts.release();
    c->bases = nb; c->starts = ns;
  }
  (void)sbytes;
  return APGK_OK;
}

int append_bases(apgk_ctx* c, const uint8_t* packed, uint64_t first_base, uint64_t n_bases) {
  if (!n_bases) return APGK_OK;
  int rc = ensure_store(c, c->total_bases + n_bases);
  if (rc) return rc;
  const uint64_t dst_bit0 = 2 * c->total_bases, src_bit0 = 2 * first_base;
  if ((dst_bit0 & 7) == 0 && (src_bit0 & 7) == 0) {
    // byte aligned on both sides: copy straight into the store
    const size_t nbytes = (size_t)((2 * n_bases + 7) / 8);
    CU(cudaMemcpyAsync(c->bases.as<uint8_t>() + (dst_bit0 >> 3), packed + (src_bit0 >> 3), nbytes,
                       cudaMemcpyHostToDevice, c->stream));
    // bits of the last byte beyond n_bases must stay zero for later appends and for the window loads
    if ((2 * n_bases) & 7) {
      // clear the tail: re-write the final partial byte masked (tiny synchronous fix-up)
      uint8_t last = packed[(src_bit0 >> 3) + nbytes - 1] & (uint8_t)((1u << ((2 * n_bases) & 7)) - 1u);
      CU(cudaMemcpyAsync(c->bases.as<uint8_t>() + (dst_bit0 >> 3) + nbytes - 1, &last, 1, cudaMemcpyHostToDevice,
                         c->stream));
      CU(cudaStreamSynchronize(c->stream));
    }
  } else {
    const uint64_t sb_byte = src_bit0 >> 3;
    const uint64_t sb_al = sb_byte & ~7ull;  // keep 8-byte alignment of the staged words
    const size_t nbytes = (size_t)(((src_bit0 + 2 * n_bases + 7) >> 3) - sb_al);
    CU(c->staging.ensure(nbytes + 32));
    CU(cudaMemsetAsync((uint8_t*)c->staging.p + (nbytes & ~(size_t)7), 0, 24, c->stream));
    CU(cudaMemcpyAsync(c->staging.p, packed + sb_al, nbytes, cudaMemcpyHostToDevice, c->stream));
    const uint64_t nbits = 2 * n_bases;
    const uint64_t nwords = ((dst_bit0 + nbits + 63) >> 6) - (dst_bit0 >> 6);
    k_append_bits<<<(unsigned)((nwords + 255) / 256), 256, 0, c->stream>>>(
        c->staging.as<uint64_t>(), src_bit0 - sb_al * 8, c->bases.as<uint64_t>(), dst_bit0, nbits);
    LAUNCHED();
  }
  return APGK_OK;
}

void invalidate_results(apgk_ctx* c) {
  c->finished = false; c->have_table = false; c->spec_loaded = false;
  c->table_from_reads = false; c->have_occ = false; c->n_occ = 0;
  c->n_instances = c->n_distinct = 0;
  c->owner_ranks = 0;
  c->part_ready = false; c->part_n = 0;
}

// ---------------------------------------------------------------- the pipeline
enum RunMode { RUN_FULL = 0, RUN_PARTITION = 1 };
template <int W, typename ElemB>
int run_levels(apgk_ctx* c, const Key<W>* dev_keys, uint64_t n_keys, RunMode mode);
template <int W, typename ElemB>
int count_buckets(apgk_ctx* c, uint64_t Nr, uint64_t N_all, uint64_t& n_prev, Key<W>* tmp_keys, bool nosync);

// k-mer instances a run over the read store sees: exact, accumulated at ingest (a read of L bases yields
// max(0, L-K+1) windows), so the host sizes buffers and grids without waiting for the level-0 histogram
uint64_t window_upper(const apgk_ctx* c) { return c->n_windows; }

// Geometry of a run over `upper` instances (forced_P > 0 overrides the choice: ranks of a sharded run
// must agree on it).  Returns true when level 1 stores 32-bit remainders.
template <int W>
bool select_geometry(apgk_ctx* c, uint64_t upper, int forced_P) {
  // decide element type of the level-1 buffer first (it fixes LOCAL_MAX, which fixes P)
  int lm_u32 = LM_U32;
  if (const char* e = getenv("APGK_LM")) { if (atoi(e) >= 256 && atoi(e) <= 12288) lm_u32 = atoi(e); }
  if (upper == 0) upper = 1;
  if (forced_P > 0) {
    make_geom(c, std::max(2, std::min(24, forced_P)));
    return W == 1 && c->geom.REM <= 32;
  }
  // try the 32-bit-remainder geometry first: one-word keys whose remainder below the prefix fits 31 bits
  int P = choose_prefix_bits(c, upper, lm_u32, true);
  make_geom(c, P);
  if (W == 1 && c->cfg.prefix_bits <= 0 && !getenv("APGK_PREFIX_BITS")) {
    while (c->geom.REM > 31 && c->geom.REM <= 34 && P < 24) make_geom(c, ++P);  // a few more prefix bits buy the fast path
  }
  const bool u32 = (W == 1 && c->geom.REM <= 32);
  if (!u32) {
    // k_local4 splits oversize ranges, so the average bucket may sit near its table's capacity
    P = use_local4(W) ? choose_prefix_bits(c, upper, LM_KEY4 * 3 / 4, true) : choose_prefix_bits(c, upper, Geo<W>::LM_KEY, false);
    make_geom(c, P);
  }
  return u32;
}

template <int W> int compact_table(apgk_ctx* c, uint64_t total);

// The result block: a few words the kernels of a step leave for the host, fetched with ONE copy at the
// step's final synchronisation (RES_* index c->res, 16 x u64 on the device, mirrored in pinned host memory).
enum { RES_RANGE_N = 0, RES_SUM_TOT0 = 1, RES_FLAGS = 2, RES_DISTINCT = 3, RES_TABLE_OVF = 4, RES_XFLAGS = 5, RES_WORDS = 16 };

int fetch_results(apgk_ctx* c) {
  CU(cudaMemcpyAsync(c->res_host, c->res.p, RES_WORDS * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return APGK_OK;
}

// The step's one synchronisation: fetch the result block, check what the kernels flagged, and settle the table
// of a single-round step that was compacted optimistically into the buffers of the previous step.
int step_epilogue(apgk_ctx* c, bool full) {
  { int r2 = fetch_results(c); if (r2) return r2; }
  if (c->res_host[RES_FLAGS] & 1ull) FAIL(APGK_E_RANGE, "a level-0 bucket holds 2^32 or more k-mers");
  if (c->res_host[RES_SUM_TOT0] && c->res_host[RES_SUM_TOT0] != c->n_windows_run)
    FAIL(APGK_E_STATE, "internal: level-0 histogram counts %llu k-mers, the input holds %llu",
         (unsigned long long)c->res_host[RES_SUM_TOT0], (unsigned long long)c->n_windows_run);
  if (full && c->table_pending) {
    c->table_pending = false;
    const uint64_t total = c->res_host[RES_DISTINCT];
    if (c->res_host[RES_TABLE_OVF]) {   // it did not fit: grow and compact again (the temp records are still in place)
      int rc = APGK_E_ARG;
      switch (c->W) {
        case 1: rc = compact_table<1>(c, total); break;
        case 2: rc = compact_table<2>(c, total); break;
        case 3: rc = compact_table<3>(c, total); break;
      }
      if (rc) return rc;
      CU(cudaStreamSynchronize(c->stream));
    }
    c->n_distinct = total;
  }
  return APGK_OK;
}

template <int W>
int finish_impl(apgk_ctx* c, const Key<W>* dev_keys, uint64_t n_keys, RunMode mode = RUN_FULL, int forced_P = 0) {
  invalidate_results(c);
  stages_reset(c);
  select_geometry<W>(c, dev_keys ? n_keys : window_upper(c), forced_P);
  if (!c->res_host) CU(cudaHostAlloc((void**)&c->res_host, RES_WORDS * 8, cudaHostAllocDefault));
  CU(c->res.ensure(RES_WORDS * 8));
  CU(cudaMemsetAsync(c->res.p, 0, RES_WORDS * 8, c->stream));
  stage_begin(c, ST_TOTAL);
  int rc;
  if constexpr (W == 1) {
    if (c->geom.REM <= 32) rc = run_levels<W, uint32_t>(c, dev_keys, n_keys, mode);
    else rc = run_levels<W, Key<W>>(c, dev_keys, n_keys, mode);
  } else {
    rc = run_levels<W, Key<W>>(c, dev_keys, n_keys, mode);
  }
  if (rc) {   // leave the context in a state the next call can start from: nothing in flight, no half-recorded intervals
    if (c->n_slices && c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    c->n_slices = 0;
    cudaStreamSynchronize(c->stream);
    c->n_ivs = 0; c->table_pending = false;
    return rc;
  }
  stage_end(c, ST_TOTAL);
  c->n_deferred = 0;
  if (mode == RUN_FULL && c->deferred.p && c->n_instances)
    CU(cudaMemcpyAsync(&c->n_deferred, c->deferred.p, 4, cudaMemcpyDeviceToHost, c->stream));
  { int r2 = step_epilogue(c, mode == RUN_FULL); if (r2) return r2; }   // the step's one synchronisation
  stages_collect(c);
  if (mode == RUN_FULL) c->finished = true;
  else c->part_ready = true;
  return APGK_OK;
}

template <typename ElemB, int W>
struct ScatterSel {  // level-1 scatter kernel: Key<W> in, ElemB out
  static auto kernel() { return k_scatter_keys<Key<W>, ElemB, Geo<W>::NT1, DIGIT_BITS, false>; }
};

// u64 accumulate: dst[i] += src[i]   (global bucket index = sum of the rounds' local prefixes)
__global__ void k_accumulate_u64(unsigned long long* __restrict__ dst, const unsigned long long* __restrict__ src, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] += src[i];
}

// grow a result buffer, keeping its first keep_bytes
int ensure_preserve(apgk_ctx* c, DevBuf& b, size_t bytes, size_t keep_bytes) {
  if (bytes <= b.cap) return APGK_OK;
  if (!keep_bytes || !b.p) { CU(b.ensure(bytes)); return APGK_OK; }
  DevBuf nb;
  if (nb.ensure(std::max(bytes, b.cap + b.cap / 2)) != cudaSuccess) {
    cudaGetLastError();
    CU(nb.ensure(bytes));   // no room for growth in steps: exactly what is needed
  }
  CU(cudaMemcpyAsync(nb.p, b.p, keep_bytes, cudaMemcpyDeviceToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  b.release();
  b = nb;
  return APGK_OK;
}

// dynamic shared memory opt-in and occupancy of a kernel: asked once per (kernel, shared bytes), not per step
template <typename K>
int kernel_setup(apgk_ctx* c, K kernel, int nt, size_t smem, int* occ_out) {
  const auto key = std::make_pair((const void*)kernel, smem);
  auto it = c->kattr.find(key);
  if (it == c->kattr.end()) {
    if (smem > 48 * 1024) CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 1;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, nt, smem));
    it = c->kattr.emplace(key, std::max(occ, 1)).first;
  }
  if (occ_out) *occ_out = it->second;
  return APGK_OK;
}

// chunk length (in tiles) of a pass whose segments hold about avg_tiles tiles each: a scatter CTA walks one
// chunk; ~4+ chunks per segment keep the CTAs balanced (the fullest canonical prefixes hold ~2x the average)
int chunk_tiles_for(uint64_t avg_tiles) {
  int ct = (int)std::min<uint64_t>((2 * avg_tiles + 3) / 4, 128);
  ct = std::max(8, ct);
  if (const char* e = getenv("APGK_CT")) { if (atoi(e) > 0) ct = atoi(e); }  // tuning knob
  return ct;
}

// ---- level 0, histogram: reads (or a key array) -> chunksum0, level-0 bucket totals tot0_dev.  The plan
// depends on the input size alone and is kept from step to step.
template <int W>
int level0_hist(apgk_ctx* c, const Key<W>* dev_keys, uint64_t n_keys, DigitFn<DIGIT_BITS>& dg0) {
  const KeyGeom g = c->geom;
  const int bins0 = 1 << g.D0;
  const uint32_t tile0 = dev_keys ? Geo<W>::TILE1 : (uint32_t)Geo<W>::NT0 * POS_PER_THREAD;
  const uint64_t n_elems = dev_keys ? n_keys : c->total_bases;
  HostPlan& hp0 = c->hp0;
  if (c->hp0_elems != n_elems || c->hp0_tile != tile0 || hp0.lp.bins != bins0 || !c->plan0.p) {
    std::vector<uint64_t> one{n_elems};
    build_plan(hp0, one, tile0, bins0);
    const size_t S1 = hp0.seg_tile0.size();
    CU(c->plan0.ensure(S1 * 16 + 64));
    unsigned char* d = c->plan0.as<unsigned char>();
    // (pageable host memory: cudaMemcpyAsync returns once the bytes are staged, and hp0 lives in the context)
    CU(cudaMemcpyAsync(d, hp0.seg_start.data(), S1 * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d + S1 * 8, hp0.seg_tile0.data(), S1 * 4, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d + S1 * 12, hp0.seg_chunk0.data(), S1 * 4, cudaMemcpyHostToDevice, c->stream));
    hp0.lp.seg_start = (const uint64_t*)d;
    hp0.lp.seg_tile0 = (const uint32_t*)(d + S1 * 8);
    hp0.lp.seg_chunk0 = (const uint32_t*)(d + S1 * 12);
    c->hp0_elems = n_elems; c->hp0_tile = tile0;
  }
  CU(c->chunksum0.ensure((size_t)hp0.lp.n_chunks * bins0 * 4));
  stage_begin(c, ST_HIST0);
  if (dev_keys) {
    k_hist_keys<Key<W>, Geo<W>::NT1, DIGIT_BITS><<<hp0.lp.n_chunks, Geo<W>::NT1, bins0 * 4, c->stream>>>(
        dev_keys, hp0.lp, dg0, c->chunksum0.as<uint32_t>());
  } else {
    // cheap formulation when the digit is a clean prefix of the real k-mer (no left padding, <= 8 bases)
    const int top_bits = (g.pad == 0 && g.D0 <= 16 && c->cfg.K >= (g.D0 + 1) / 2 && !getenv("APGK_NO_TOPDIGITS")) ? g.D0 : 0;
    if (c->n_slices == 0) {
      k_hist_reads<W, Geo<W>::NT0, DIGIT_BITS><<<hp0.lp.n_chunks, Geo<W>::NT0, bins0 * 4, c->stream>>>(
          read_store(c), dg0, hp0.lp, top_bits, c->chunksum0.as<uint32_t>());
    } else {
      // streamed ingest: the chunks whose windows lie inside the slices that have landed, slice after slice
      const uint64_t reach = (uint64_t)c->cfg.K + 256;  // a window start reads at most K + 48 bases ahead
      uint32_t c_lo = 0;
      for (size_t i = 0; i < c->n_slices; i++) {
        CU(cudaStreamWaitEvent(c->stream, c->slice_ev[i], 0));
        uint32_t c_hi = hp0.lp.n_chunks;
        if (i + 1 < c->n_slices) {
          const uint64_t safe = c->slice_end[i] > reach ? c->slice_end[i] - reach : 0;
          c_hi = (uint32_t)std::min<uint64_t>(hp0.lp.n_chunks, safe / ((uint64_t)tile0 * hp0.lp.chunk_tiles));
        }
        if (c_hi > c_lo) {
          k_hist_reads<W, Geo<W>::NT0, DIGIT_BITS><<<c_hi - c_lo, Geo<W>::NT0, bins0 * 4, c->stream>>>(
              read_store(c), dg0, hp0.lp, top_bits, c->chunksum0.as<uint32_t>(), c_lo);
          c->launches++;
          c_lo = c_hi;
        }
      }
      c->n_slices = 0;
    }
  }
  LAUNCHED();
  stage_end(c, ST_HIST0);
  stage_begin(c, ST_SCAN0);
  CU(c->tot0_dev.ensure((size_t)bins0 * 8));
  CU(c->bstart32.ensure((size_t)bins0 * 4));
  k_segscan<COL_NT><<<1, COL_NT, 0, c->stream>>>(hp0.lp, c->chunksum0.as<uint32_t>(), c->tot0_dev.as<unsigned long long>(),
                                                 c->bstart32.as<uint32_t>(), nullptr, 0);
  LAUNCHED();
  stage_end(c, ST_SCAN0);
  return APGK_OK;
}

// ---- level 0, scatter of the level-0 buckets [lo, hi) (all of them: no filtering) -> A, bucketed by D0 bits
template <int W>
int level0_scatter(apgk_ctx* c, const Key<W>* dev_keys, DigitFn<DIGIT_BITS> dg0, int lo, int hi, uint64_t n_round) {
  const KeyGeom g = c->geom;
  const int bins0 = 1 << g.D0;
  const bool filter = lo > 0 || hi < bins0;
  const HostPlan& hp0 = c->hp0;
  const uint32_t tile0 = hp0.lp.tile_elems;
  CU(c->A.ensure(std::max<size_t>(n_round, 1) * sizeof(Key<W>)));
  CU(c->bstart64.ensure(((size_t)bins0 + 1) * 8));
  stage_begin(c, ST_SCAN0);
  // starts of the round's level-0 buckets in A; also the histogram's grand total and the 2^32 check -> result block
  k_plan_range<<<1, PLAN_NT, 0, c->stream>>>(c->tot0_dev.as<unsigned long long>(), bins0, lo, hi, 1u, 1u,
                                            c->bstart64.as<unsigned long long>(), nullptr, nullptr, c->res.as<unsigned long long>());
  LAUNCHED();
  stage_end(c, ST_SCAN0);
  dg0.flo = (uint32_t)lo; dg0.fwidth = (uint32_t)(hi - lo);
  stage_begin(c, ST_SCATTER0);
  const size_t sm = scatter_smem_bytes<Key<W>>(tile0, bins0);
  if (dev_keys) {
    auto launch = [&](auto kern) -> int {
      { int rc = kernel_setup(c, kern, Geo<W>::NT1, sm, nullptr); if (rc) return rc; }
      kern<<<hp0.lp.n_chunks, Geo<W>::NT1, sm, c->stream>>>(dev_keys, hp0.lp, dg0, c->chunksum0.as<uint32_t>(),
                                                            c->bstart64.as<uint64_t>(), 0, 0, c->A.as<Key<W>>());
      return APGK_OK;
    };
    int rc = filter ? launch(k_scatter_keys<Key<W>, Key<W>, Geo<W>::NT1, DIGIT_BITS, true>)
                    : launch(k_scatter_keys<Key<W>, Key<W>, Geo<W>::NT1, DIGIT_BITS, false>);
    if (rc) return rc;
  } else {
    auto launch = [&](auto kern) -> int {
      { int rc = kernel_setup(c, kern, Geo<W>::NTS, sm, nullptr); if (rc) return rc; }
      kern<<<hp0.lp.n_chunks, Geo<W>::NTS, sm, c->stream>>>(read_store(c), dg0, hp0.lp, c->chunksum0.as<uint32_t>(),
                                                            c->bstart64.as<uint64_t>(), c->A.as<Key<W>>());
      return APGK_OK;
    };
    int rc = filter ? launch(k_scatter_reads<W, Geo<W>::NTS, DIGIT_BITS, true, Geo<W>::NPOS>)
                    : launch(k_scatter_reads<W, Geo<W>::NTS, DIGIT_BITS, false, Geo<W>::NPOS>);
    if (rc) return rc;
  }
  LAUNCHED();
  stage_end(c, ST_SCATTER0);
  return APGK_OK;
}

// ---- level 1 over the level-0 buckets (segments) [s_lo, s_hi), whose n_range keys start at a_src:
// -> B (n_range elements bucketed by D0+D1 bits, relative to the range), bucket sizes segtot, offsets bofs.
// The plan (tiles / chunks of every segment) is made on the device from tot0_dev; the host only bounds the grid.
// d2 > 0 also leaves the sizes of the 2^d2 sub-buckets of every bucket in sub_sizes (sharded exchange).
template <int W, typename ElemB>
int level1(apgk_ctx* c, int s_lo, int s_hi, uint64_t n_range, const Key<W>* a_src, int d2) {
  const KeyGeom g = c->geom;
  const int bins0 = 1 << g.D0, bins1 = 1 << g.D1;
  const uint32_t tile = Geo<W>::TILE1;
  const int n_seg_in = std::max(1, s_hi - s_lo);
  const int ct = chunk_tiles_for(n_range / tile / (uint64_t)n_seg_in);
  const uint64_t tiles_bound = n_range / tile + (uint64_t)n_seg_in;
  const uint32_t chunks_bound = (uint32_t)(tiles_bound / (uint64_t)ct + (uint64_t)n_seg_in + 1);
  const size_t S1 = (size_t)bins0 + 1;
  CU(c->plan.ensure(S1 * 16 + 64));
  unsigned char* d = c->plan.as<unsigned char>();
  LevelPlan lp{};
  lp.bins = bins1; lp.n_segments = bins0; lp.chunk_tiles = ct; lp.tile_elems = tile;
  lp.n_tiles = (uint32_t)tiles_bound; lp.n_chunks = chunks_bound;
  lp.seg_start = (const uint64_t*)d;
  lp.seg_tile0 = (const uint32_t*)(d + S1 * 8);
  lp.seg_chunk0 = (const uint32_t*)(d + S1 * 12);
  DigitSpec ds1{DIGIT_BITS, g.TB - g.D0 - g.D1, g.D1, g.pad, 0};
  const DigitFn<DIGIT_BITS> dg1 = make_digit_fn<DIGIT_BITS>(ds1);
  DigitSpec dsw{DIGIT_BITS, g.TB - g.D0 - g.D1 - d2, g.D1 + d2, g.pad, 0};
  const DigitFn<DIGIT_BITS> dgw = make_digit_fn<DIGIT_BITS>(dsw);
  stage_begin(c, ST_SCAN1);
  k_plan_range<<<1, PLAN_NT, 0, c->stream>>>(c->tot0_dev.as<unsigned long long>(), bins0, s_lo, s_hi, tile, (uint32_t)ct,
                                            (unsigned long long*)d, (uint32_t*)(d + S1 * 8), (uint32_t*)(d + S1 * 12), nullptr);
  LAUNCHED();
  stage_end(c, ST_SCAN1);
  CU(c->chunksum.ensure((size_t)chunks_bound * bins1 * 4));
  CU(c->segtot.ensure((size_t)c->nb1 * 8));
  CU(c->bstart32.ensure((size_t)c->nb1 * 4));
  CU(c->bofs.ensure(((size_t)c->nb1 + 1) * 8));
  if (d2 > 0) {
    CU(c->sub_sizes.ensure(((size_t)c->nb1 << d2) * 4 + 16));
    CU(cudaMemsetAsync(c->sub_sizes.p, 0, ((size_t)c->nb1 << d2) * 4, c->stream));
  }
  stage_begin(c, ST_HIST1);
  {
    auto kern = k_hist_keys<Key<W>, Geo<W>::NT1, DIGIT_BITS>;
    const size_t smh = ((size_t)bins1 << d2) * 4;
    { int rc = kernel_setup(c, kern, Geo<W>::NT1, smh, nullptr); if (rc) return rc; }
    kern<<<chunks_bound, Geo<W>::NT1, smh, c->stream>>>(a_src, lp, dg1, c->chunksum.as<uint32_t>(), dgw, d2,
                                                        d2 > 0 ? c->sub_sizes.as<uint32_t>() : nullptr);
    LAUNCHED();
  }
  stage_end(c, ST_HIST1);
  stage_begin(c, ST_SCAN1);
  k_segscan<COL_NT><<<bins0, COL_NT, 0, c->stream>>>(lp, c->chunksum.as<uint32_t>(), c->segtot.as<unsigned long long>(),
                                                     c->bstart32.as<uint32_t>(), c->bofs.as<unsigned long long>(), 1);
  LAUNCHED();
  stage_end(c, ST_SCAN1);
  CU(c->B.ensure(std::max<size_t>(n_range, 1) * sizeof(ElemB) + 16));
  stage_begin(c, ST_SCATTER1);
  {
    // APGK_BULK=1: the TMA bulk write-out (k_scatter_keys_bulk) for 32-bit remainders.  Off by default: measured
    // slower than the register write-out (profiles/r02_bulk_scatter.txt: 23.3 against 19.7 ms) -- the element-wise
    // write-out doubles as the work that hides the next tile's load latency, and a tile's 1 024 copies of ~64 bytes
    // do not buy back what that costs.  Kept (and tested) as the measured alternative.
    const char* eb = getenv("APGK_BULK");
    const bool bulk = eb && !strcmp(eb, "1");
    const size_t smb = scatter_bulk_smem_bytes<ElemB>(tile, bins1);
    if (bulk && sizeof(ElemB) == 4 && smb <= 200 * 1024 && bins1 <= Geo<W>::NT1) {
      auto kern = k_scatter_keys_bulk<Key<W>, ElemB, Geo<W>::NT1, DIGIT_BITS, false>;
      { int rc = kernel_setup(c, kern, Geo<W>::NT1, smb, nullptr); if (rc) return rc; }
      kern<<<chunks_bound, Geo<W>::NT1, smb, c->stream>>>(a_src, lp, dg1, c->chunksum.as<uint32_t>(), nullptr, g.pad, g.REM,
                                                          c->B.as<ElemB>());
    } else {
      auto kern = ScatterSel<ElemB, W>::kernel();
      const size_t sm = scatter_smem_bytes<Key<W>>(tile, bins1);
      { int rc = kernel_setup(c, kern, Geo<W>::NT1, sm, nullptr); if (rc) return rc; }
      kern<<<chunks_bound, Geo<W>::NT1, sm, c->stream>>>(a_src, lp, dg1, c->chunksum.as<uint32_t>(), nullptr, g.pad, g.REM,
                                                         c->B.as<ElemB>());
    }
    LAUNCHED();
  }
  stage_end(c, ST_SCATTER1);
  return APGK_OK;
}

// device memory the temp buffers of a run may take: what is free now plus what the context already holds for them
int temp_budget(apgk_ctx* c, size_t* budget) {
  size_t fr = 0, tot = 0;
  CU(cudaMemGetInfo(&fr, &tot));
  const size_t held = c->A.cap + c->B.cap + c->T.cap;  // reusable
  *budget = (size_t)((double)(fr + held) * 0.60);       // temp buffers ~60 % of it; the result table gets the rest
  return APGK_OK;
}

template <int W, typename ElemB>
int run_levels(apgk_ctx* c, const Key<W>* dev_keys, uint64_t n_keys, RunMode mode) {
  const KeyGeom g = c->geom;
  const int bins0 = 1 << g.D0, bins1 = 1 << g.D1;
  int local_max = std::is_same<ElemB, uint32_t>::value ? LM_U32 : (use_local4(W) ? LM_KEY4 : Geo<W>::LM_KEY);
  if (std::is_same<ElemB, uint32_t>::value) {  // tuning knob
    if (const char* e = getenv("APGK_LM")) { if (atoi(e) >= 256 && atoi(e) <= 12288) local_max = atoi(e); }
  }
  const int want_table = (c->cfg.flags & APGK_WANT_COUNTS) ? 1 : 0;
  c->elem_bytes = sizeof(ElemB);
  c->local_max = (uint32_t)local_max;
  c->nb1 = (uint32_t)bins0 * (uint32_t)bins1;
  c->n_rounds = 0; c->n_big = 0; c->n_distinct = 0;
  c->table_pending = false;
  CU(c->spec_dense.ensure((size_t)SPEC_DENSE * 8));
  CU(cudaMemsetAsync(c->spec_dense.p, 0, (size_t)SPEC_DENSE * 8, c->stream));
  CU(c->out_off.ensure(((size_t)c->nb1 + 1) * 8));
  CU(cudaMemsetAsync(c->out_off.p, 0, ((size_t)c->nb1 + 1) * 8, c->stream));
  const uint64_t N = dev_keys ? n_keys : c->n_windows;   // exact, known before any kernel runs
  c->n_instances = N; c->n_windows_run = N;
  c->tot0_host.assign((size_t)bins0, 0);
  if (N == 0) {  // nothing to count
    { int rc = wait_ingest(c); if (rc) return rc; }
    c->have_table = want_table != 0;
    c->part_n = 0;
    if (mode == RUN_PARTITION) {
      CU(c->segtot.ensure((size_t)c->nb1 * 8));
      CU(cudaMemsetAsync(c->segtot.p, 0, (size_t)c->nb1 * 8, c->stream));
    }
    return APGK_OK;
  }

  // ================= level 0: one histogram pass over everything (all rounds share it)
  DigitSpec ds0{DIGIT_BITS, g.TB - g.D0, g.D0, g.pad, 0};
  DigitFn<DIGIT_BITS> dg0 = make_digit_fn<DIGIT_BITS>(ds0);
  { int rc = level0_hist<W>(c, dev_keys, n_keys, dg0); if (rc) return rc; }

  // ================= rounds over k-mer space (SortKmers "passes" / KmerParcels "parcels").  Two levels:
  //   outer rounds  consecutive level-0 buckets whose full keys (A) fit: one (filtered) level-0 scatter each
  //   inner rounds  sub-ranges of an outer round whose level-1 copy + temp counts (B, T) fit: level 1 + counting
  // so a memory-tight run re-extracts the reads once per OUTER round only.  The common case -- everything
  // fits at once -- needs nothing from the device to be planned: no host round trip.
  const size_t eA = sizeof(Key<W>), eB = sizeof(ElemB) + (want_table ? 4 : 0);
  uint64_t cap_outer = c->cfg.max_round_keys, cap_inner = c->cfg.max_inner_keys;
  if (const char* e = getenv("APGK_ROUND_KEYS")) { if (atoll(e) > 0) cap_outer = (uint64_t)atoll(e); }
  if (const char* e = getenv("APGK_INNER_KEYS")) { if (atoll(e) > 0) cap_inner = (uint64_t)atoll(e); }
  bool single;
  if (cap_outer) {
    if (!cap_inner) cap_inner = cap_outer;
    single = N <= cap_outer && N <= cap_inner;
    c->last_cap_keys = std::min(cap_outer, cap_inner);
  } else {
    single = N * (eA + eB) <= c->A.cap + c->B.cap + c->T.cap && N * eA <= c->A.cap && N * sizeof(ElemB) <= c->B.cap;
    if (!single || mode == RUN_PARTITION) {
      size_t budget = 0;
      { int rc = temp_budget(c, &budget); if (rc) return rc; }
      c->last_cap_keys = (uint64_t)(budget / (eA + eB));
      single = N <= c->last_cap_keys;
      if (!single) {
        // A holds an outer round, B + T a quarter of it (unless the caller fixed the inner size)
        const uint64_t ci = cap_inner;
        cap_outer = ci ? (budget > ci * eB ? (budget - ci * eB) / eA : 1) : (uint64_t)((double)budget / ((double)eA + (double)eB / 4.0));
        cap_inner = ci ? ci : std::max<uint64_t>(1, cap_outer / 4);
        cap_outer = std::max<uint64_t>(cap_outer, 1);
      }
    }
  }
  const bool forced_range = mode == RUN_PARTITION && c->force_d0_lo >= 0;
  struct Round { int lo, hi; uint64_t n; std::vector<std::array<uint64_t, 3>> inner; };  // inner: {s_lo, s_hi, n}
  std::vector<Round> rounds;
  std::vector<uint64_t>& tot0 = c->tot0_host;
  if (!single || mode == RUN_PARTITION) {
    // the plan needs the level-0 totals on the host: the one mid-step round trip of the memory-tight path
    CU(cudaMemcpyAsync(tot0.data(), c->tot0_dev.p, (size_t)bins0 * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    uint64_t sum = 0;
    for (int d = 0; d < bins0; d++) {
      if (tot0[d] >= (1ull << 32)) FAIL(APGK_E_RANGE, "level-0 bucket %d holds %llu k-mers (>= 2^32)", d, (unsigned long long)tot0[d]);
      sum += tot0[d];
    }
    if (sum != N) FAIL(APGK_E_STATE, "internal: level-0 histogram counts %llu k-mers, expected %llu", (unsigned long long)sum, (unsigned long long)N);
  }
  if (forced_range) {   // the caller runs the rounds (sharded counting: all ranks use the same ranges)
    Round r;
    r.lo = std::min(c->force_d0_lo, bins0); r.hi = std::min(std::max(c->force_d0_hi, c->force_d0_lo), bins0);
    r.n = 0;
    for (int d = r.lo; d < r.hi; d++) r.n += tot0[d];
    r.inner.push_back({(uint64_t)r.lo, (uint64_t)r.hi, r.n});
    rounds.push_back(r);
  } else if (single) {
    Round r{0, bins0, N, {}};
    r.inner.push_back({0, (uint64_t)bins0, N});
    rounds.push_back(r);
  } else {
    int lo = 0; uint64_t acc = 0;
    auto close_outer = [&](int hi) {
      Round r{lo, hi, acc, {}};
      int ilo = lo; uint64_t iacc = 0;
      for (int d = lo; d < hi; d++) {
        if (iacc && iacc + tot0[d] > cap_inner) { r.inner.push_back({(uint64_t)ilo, (uint64_t)d, iacc}); ilo = d; iacc = 0; }
        iacc += tot0[d];
      }
      r.inner.push_back({(uint64_t)ilo, (uint64_t)hi, iacc});
      rounds.push_back(r);
    };
    for (int d = 0; d < bins0; d++) {
      if (acc && acc + tot0[d] > cap_outer) { close_outer(d); lo = d; acc = 0; }
      acc += tot0[d];
    }
    close_outer(bins0);
  }
  for (const Round& r : rounds) c->n_rounds += (uint32_t)r.inner.size();
  if (mode == RUN_PARTITION && !forced_range && !single)
    FAIL(APGK_E_RANGE, "apgk_partition: %u k-mer-space rounds would be needed; the sharded exchange takes one", c->n_rounds);

  CU(c->spec_ovf.ensure(((size_t)N / SPEC_DENSE + 16) * 8));
  CU(cudaMemsetAsync(c->spec_ovf.p, 0, 8, c->stream));
  CU(c->nd.ensure(((size_t)c->nb1 + 1) * 4));
  CU(c->out_off_local.ensure(((size_t)c->nb1 + 1) * 8));
  CU(c->stats.ensure(64));
  uint64_t n_prev = 0;  // records already in the result table
  uint64_t n_counted = 0;  // instances of the rounds so far (the table's growth hint)

  for (const Round& r : rounds) {
    if (r.n == 0) {
      if (mode == RUN_PARTITION) {   // nothing in this range: an empty partition
        CU(c->segtot.ensure((size_t)c->nb1 * 8));
        CU(cudaMemsetAsync(c->segtot.p, 0, (size_t)c->nb1 * 8, c->stream));
        c->part_n = 0;
        return APGK_OK;
      }
      continue;
    }
    { int rc = level0_scatter<W>(c, dev_keys, dg0, r.lo, r.hi, r.n); if (rc) return rc; }
    uint64_t off_a = 0;   // keys of the outer round before the current inner range
    for (const auto& in : r.inner) {
      n_counted += in[2];
      const uint64_t n_in = in[2];
      if (n_in == 0) continue;
      Key<W>* a_src = c->A.as<Key<W>>() + off_a;
      { int rc = level1<W, ElemB>(c, (int)in[0], (int)in[1], n_in, a_src, 0); if (rc) return rc; }
      if (mode == RUN_PARTITION) { c->part_n = n_in; return APGK_OK; }
      c->count_src = c->B.p; c->bucket_lo = c->bucket_hi = 0;
      if (!single) { c->bucket_lo = (uint32_t)in[0] * (uint32_t)bins1; c->bucket_hi = (uint32_t)in[1] * (uint32_t)bins1; }  // the others are empty
      // the temp records of the range's buckets go over the range's own level-0 keys: dead once level 1 has run
      c->table_scale = single ? 1.0 : std::max(1.0, (double)N / (double)std::max<uint64_t>(n_counted, 1));
      { int rc = count_buckets<W, ElemB>(c, n_in, N, n_prev, a_src, single); if (rc) return rc; }
      c->table_scale = 1.0;
      c->bucket_lo = c->bucket_hi = 0;
      off_a += n_in;
    }
  }
  if (!single) c->n_distinct = n_prev;
  c->have_table = want_table != 0;
  return APGK_OK;
}

// final table of a single-round step whose record count is on the host: (re)size the result buffers, compact
template <int W>
int compact_table(apgk_ctx* c, uint64_t total) {
  CU(c->out_keys.ensure(std::max<size_t>(total + (total >> 5), 1) * sizeof(Key<W>)));
  CU(c->out_cnt.ensure(std::max<size_t>(total + (total >> 5), 1) * 4));
  k_compact<W><<<c->n_sm * 8, 256, 0, c->stream>>>(c->tmp_keys_last ? (const Key<W>*)c->tmp_keys_last : c->A.as<Key<W>>(), c->T.as<uint32_t>(),
                                                   c->bofs.as<unsigned long long>(), c->out_off_local.as<unsigned long long>(), c->nb1,
                                                   c->out_keys.as<Key<W>>(), c->out_cnt.as<uint32_t>(), nullptr, 0ull, nullptr);
  LAUNCHED();
  return APGK_OK;
}

// ---------------------------------------------------------------- per-bucket sort + count, table append
// Input: c->count_src holds Nr elements grouped by the nb1 buckets (offsets c->bofs, sizes c->segtot).  Appends the
// distinct k-mers of these buckets to the result table at n_prev (buckets ascend in k-mer order).  tmp_keys:
// Nr keys of scratch for the per-bucket records.  nosync (single-round steps, n_prev == 0): nothing is read
// back here -- the table is compacted into the result buffers as they are and the caller checks the result
// block (RES_DISTINCT, RES_TABLE_OVF) at the step's final synchronisation.
template <int W, typename ElemB>
int count_buckets(apgk_ctx* c, uint64_t Nr, uint64_t N, uint64_t& n_prev, Key<W>* tmp_keys, bool nosync) {
  const KeyGeom g = c->geom;
  const int local_max = (int)c->local_max;
  int l3_nt = L3_NT;
  if (std::is_same<ElemB, uint32_t>::value) {
    if (const char* e = getenv("APGK_L3_NT")) { if (atoi(e) == 256 || atoi(e) == 512) l3_nt = atoi(e); }
  }
  const bool use_l3 = std::is_same<ElemB, uint32_t>::value && g.REM >= 1 && g.REM <= 31;
  const bool use_l4 = !std::is_same<ElemB, uint32_t>::value && use_local4(W) && g.pad == 0 && g.REM >= 1;
  const int want_table = (c->cfg.flags & APGK_WANT_COUNTS) ? 1 : 0;
  // bucket classification (oversize list): the range-splitting kernels take every bucket size
  const uint32_t big_cap = (uint32_t)(Nr / local_max + 16);
  uint64_t n_big = 0;
  unsigned long long stats[2] = {0, 0};
  if (!(use_l3 || use_l4)) {
    CU(c->big_list.ensure((size_t)big_cap * 4));
    CU(cudaMemsetAsync(c->stats.p, 0, 64, c->stream));
    k_classify<<<(c->nb1 + 255) / 256, 256, 0, c->stream>>>(c->segtot.as<unsigned long long>(), c->nb1, (uint32_t)local_max,
                                                           c->big_list.as<uint32_t>(), big_cap, c->stats.as<unsigned long long>());
    LAUNCHED();
    CU(cudaMemcpyAsync(stats, c->stats.p, 16, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    n_big = stats[0];
    c->n_big += n_big;
  }
  {
    EmitCtx<W> ec;
    ec.want_table = want_table; ec.rem_bits = g.REM; ec.pad = g.pad;
    ec.tmp_keys = tmp_keys;
    c->tmp_keys_last = tmp_keys;
    if (want_table) CU(c->T.ensure(std::max<size_t>(Nr, 1) * 4));
    ec.tmp_cnt = c->T.as<uint32_t>();
    ec.spec_dense = c->spec_dense.as<unsigned long long>();
    ec.spec_ovf = c->spec_ovf.as<unsigned long long>();
    ec.spec_ovf_cap = (uint32_t)(N / SPEC_DENSE + 8);
    BucketTable bt;
    bt.bofs = c->bofs.as<unsigned long long>();
    bt.bsize = c->segtot.as<unsigned long long>();
    bt.nb = c->bucket_hi ? c->bucket_hi : c->nb1; bt.local_max = (uint32_t)local_max; bt.b0 = c->bucket_hi ? c->bucket_lo : 0;
    if (c->bucket_hi) CU(cudaMemsetAsync(c->nd.p, 0, ((size_t)c->nb1 + 1) * 4, c->stream));  // buckets outside the shard: no records
    CU(c->deferred.ensure(((size_t)c->nb1 + 1) * 4));
    CU(cudaMemsetAsync(c->deferred.p, 0, 4, c->stream));
    stage_begin(c, ST_LOCAL);
    if (use_l3) {
      // 32-bit remainders: order-preserving hash kernel; it takes every bucket size (range splitting)
      if constexpr (std::is_same<ElemB, uint32_t>::value) {
        auto launch3 = [&](auto kern3, int nt) -> int {
          const size_t sm3 = Local3Smem::bytes(local_max);
          int occ3 = 1;
          { int rc = kernel_setup(c, kern3, nt, sm3, &occ3); if (rc) return rc; }
          const uint32_t grid3 = std::min<uint32_t>(c->nb1, (uint32_t)(c->n_sm * std::max(occ3, 1)));
          kern3<<<grid3, nt, sm3, c->stream>>>((const uint32_t*)c->count_src, bt, g.REM, ec, c->nd.as<uint32_t>());
          return APGK_OK;
        };
        int rc3 = l3_nt == 256 ? launch3(k_local3<256, W>, 256) : launch3(k_local3<512, W>, 512);
        if (rc3) return rc3;
        LAUNCHED();
      }
    } else if (use_l4) {
      // full-key elements: tag-hash kernel; it takes every bucket size (range splitting)
      if constexpr (!std::is_same<ElemB, uint32_t>::value) {
        auto kern4 = k_local4<512, W>;
        const size_t sm4 = Local4Smem::bytes(local_max, W);
        int occ4 = 1;
        { int rc = kernel_setup(c, kern4, 512, sm4, &occ4); if (rc) return rc; }
        const uint32_t grid4 = std::min<uint32_t>(c->nb1, (uint32_t)(c->n_sm * std::max(occ4, 1)));
        kern4<<<grid4, 512, sm4, c->stream>>>((const Key<W>*)c->count_src, bt, g.REM, ec, c->nd.as<uint32_t>());
        LAUNCHED();
      }
    } else {
      // general element types: warp-table kernel; buckets it cannot take land on the deferred list ...
      auto kern2 = k_local2<ElemB, W>;
      const size_t sm2 = Local2Smem<ElemB>::bytes(local_max);
      int occ2 = 1;
      { int rc = kernel_setup(c, kern2, L2_NT, sm2, &occ2); if (rc) return rc; }
      const uint32_t grid2 = std::min<uint32_t>(c->nb1, (uint32_t)(c->n_sm * std::max(occ2, 1)));
      kern2<<<grid2, L2_NT, sm2, c->stream>>>((const ElemB*)c->count_src, bt, g.REM, ec, c->nd.as<uint32_t>(),
                                              c->deferred.as<uint32_t>(), c->nb1);
      LAUNCHED();
      // ... which the barrier-heavy general kernel then walks (normally empty)
      auto kern = k_local<ElemB, W>;
      const size_t sm = LocalSmem<ElemB>::bytes(local_max);
      int occ = 1;
      { int rc = kernel_setup(c, kern, LOCAL_NT, sm, &occ); if (rc) return rc; }
      const uint32_t grid = std::min<uint32_t>(c->nb1, (uint32_t)(c->n_sm * std::max(occ, 1)));
      kern<<<grid, LOCAL_NT, sm, c->stream>>>((const ElemB*)c->count_src, bt, g.REM, ec, c->nd.as<uint32_t>(),
                                              c->deferred.as<uint32_t>(), c->nb1);
      LAUNCHED();
    }
    stage_end(c, ST_LOCAL);
    if (n_big) {
      if (n_big > big_cap) FAIL(APGK_E_RANGE, "internal: oversize bucket list overflow");
      auto kern = k_big<ElemB, W>;
      const size_t sm = LocalSmem<ElemB>::bytes(local_max);
      int occ = 1;
      { int rc = kernel_setup(c, kern, LOCAL_NT, sm, &occ); if (rc) return rc; }
      const uint32_t grid = (uint32_t)std::min<uint64_t>(n_big, (uint64_t)c->n_sm * std::max(occ, 1));
      CU(c->scratch.ensure((size_t)stats[1] * sizeof(ElemB) + 16));
      CU(c->stacks.ensure((size_t)grid * BIG_STACK * 16));
      CU(c->misc.ensure(64));
      CU(cudaMemsetAsync(c->misc.p, 0, 64, c->stream));
      BigParams bp;
      bp.big_list = c->big_list.as<uint32_t>();
      bp.n_big = (const uint32_t*)c->stats.p;  // low word of stats[0]
      bp.ticket = c->misc.as<unsigned int>();
      bp.scratch_cursor = (unsigned long long*)(c->misc.as<unsigned char>() + 8);
      bp.scratch = c->scratch.p;
      bp.stacks = c->stacks.as<unsigned long long>();
      stage_begin(c, ST_BIG);
      kern<<<grid, LOCAL_NT, sm, c->stream>>>((ElemB*)c->count_src, bt, g.REM, ec, c->nd.as<uint32_t>(), bp);
      LAUNCHED();
      stage_end(c, ST_BIG);
    }

    // ---- table: this round's records are appended (rounds ascend in k-mer space, so the table stays sorted)
    stage_begin(c, ST_TABLE);
    {
      const uint64_t n = c->nb1;
      const uint32_t nblocks = (uint32_t)((n + 1 + SCAN_BLOCK - 1) / SCAN_BLOCK);
      CU(c->blocksum.ensure(((size_t)nblocks + 1) * 8));
      unsigned long long* res = c->res.as<unsigned long long>();
      k_scan_blocksum<<<nblocks, SCAN_NT, 0, c->stream>>>(c->nd.as<uint32_t>(), n, c->blocksum.as<unsigned long long>());
      LAUNCHED();
      k_scan_top<<<1, SCAN_NT, 0, c->stream>>>(c->blocksum.as<unsigned long long>(), nblocks, res ? res + RES_DISTINCT : nullptr);
      LAUNCHED();
      k_scan_apply<<<nblocks, SCAN_NT, 0, c->stream>>>(c->nd.as<uint32_t>(), n, c->blocksum.as<unsigned long long>(),
                                                       c->out_off_local.as<unsigned long long>());
      LAUNCHED();
      // global prefix index = sum over rounds of the local prefixes (buckets outside a round add 0 / its total)
      k_accumulate_u64<<<(unsigned)((n + 1 + 255) / 256), 256, 0, c->stream>>>(c->out_off.as<unsigned long long>(),
                                                                              c->out_off_local.as<unsigned long long>(), n + 1);
      LAUNCHED();
      const bool optimistic = nosync && n_prev == 0 && (!want_table || (c->out_keys.cap && c->out_cnt.cap));
      if (optimistic) {
        if (want_table) {
          const unsigned long long cap = std::min<unsigned long long>(c->out_keys.cap / sizeof(Key<W>), c->out_cnt.cap / 4);
          k_compact<W><<<c->n_sm * 8, 256, 0, c->stream>>>(tmp_keys, c->T.as<uint32_t>(), c->bofs.as<unsigned long long>(),
                                                           c->out_off_local.as<unsigned long long>(), c->nb1, c->out_keys.as<Key<W>>(),
                                                           c->out_cnt.as<uint32_t>(), res + RES_DISTINCT, cap, res + RES_TABLE_OVF);
          LAUNCHED();
        }
        c->table_pending = true;   // finish_impl reads RES_DISTINCT / RES_TABLE_OVF at the step's synchronisation
      } else {
        unsigned long long total = 0;
        CU(cudaMemcpyAsync(&total, c->blocksum.as<unsigned long long>() + nblocks, 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        if (want_table) {
          // a little slack when this is the whole table (the next step reuses the buffers); when it grows round by
          // round, room for the rounds still to come (table_scale: all instances over those counted so far), so that
          // it is allocated once, while it is small, and not copied again and again
          size_t want = n_prev + total + (nosync ? (total >> 5) : 0);
          if (!nosync && c->table_scale > 1.0 && (c->out_keys.cap < want * sizeof(Key<W>) || c->out_cnt.cap < want * 4))
            want = (size_t)((double)want * c->table_scale * 1.12) + 1024;
          { int rc = ensure_preserve(c, c->out_keys, std::max<size_t>(want, 1) * sizeof(Key<W>), n_prev * sizeof(Key<W>)); if (rc) return rc; }
          { int rc = ensure_preserve(c, c->out_cnt, std::max<size_t>(want, 1) * 4, n_prev * 4); if (rc) return rc; }
          k_compact<W><<<c->n_sm * 8, 256, 0, c->stream>>>(tmp_keys, c->T.as<uint32_t>(), c->bofs.as<unsigned long long>(),
                                                           c->out_off_local.as<unsigned long long>(), c->nb1,
                                                           c->out_keys.as<Key<W>>() + n_prev, c->out_cnt.as<uint32_t>() + n_prev,
                                                           nullptr, 0ull, nullptr);
          LAUNCHED();
        }
        n_prev += total;
        if (nosync) c->n_distinct = n_prev;
      }
    }
    stage_end(c, ST_TABLE);
    }
  return APGK_OK;
}

int load_spectrum(apgk_ctx* c) {
  if (c->spec_loaded) return APGK_OK;
  if (!c->finished) FAIL(APGK_E_STATE, "apgk_finish has not run");
  std::vector<uint64_t> dense(SPEC_DENSE, 0);
  c->sparse_f.clear(); c->sparse_n.clear(); c->spec_host.clear();
  std::vector<uint64_t> ovf;
  if (c->n_instances) {
    CU(cudaMemcpyAsync(dense.data(), c->spec_dense.p, (size_t)SPEC_DENSE * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (c->spec_ovf.p) {
      unsigned long long n_ovf = 0;
      CU(cudaMemcpyAsync(&n_ovf, c->spec_ovf.p, 8, cudaMemcpyDeviceToHost, c->stream));
      CU(cudaStreamSynchronize(c->stream));
      if (n_ovf) {
        ovf.resize(n_ovf);
        CU(cudaMemcpyAsync(ovf.data(), (unsigned long long*)c->spec_ovf.p + 1, n_ovf * 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        std::sort(ovf.begin(), ovf.end());
      }
    }
  }
  for (uint64_t f = 1; f < SPEC_DENSE; f++)
    if (dense[f]) { c->sparse_f.push_back(f); c->sparse_n.push_back(dense[f]); }
  for (size_t i = 0; i < ovf.size();) {
    size_t j = i;
    while (j < ovf.size() && ovf[j] == ovf[i]) j++;
    c->sparse_f.push_back(ovf[i]); c->sparse_n.push_back(j - i);
    i = j;
  }
  c->spec_loaded = true;
  return APGK_OK;
}

template <int W>
FreqTable<W> freq_table(const apgk_ctx* c) {
  FreqTable<W> t;
  t.keys = c->out_keys.as<Key<W>>();
  t.counts = c->out_cnt.as<uint32_t>();
  t.index = c->out_off.as<unsigned long long>();
  t.nb = c->nb1;
  t.prefix_pos = c->geom.REM; t.prefix_len = c->geom.D0 + c->geom.D1; t.pad = c->geom.pad; t.D1 = c->geom.D1;
  return t;
}

template <int W>
int lookup_impl(apgk_ctx* c, const uint64_t* kmers, uint64_t n, int canon, uint32_t* out) {
  if (!n) return APGK_OK;
  struct Tmp { DevBuf b; ~Tmp() { b.release(); } } q_, r_;   // released on every path out
  DevBuf& q = q_.b; DevBuf& r = r_.b;
  CU(q.ensure(n * sizeof(Key<W>)));
  CU(r.ensure(n * 4));
  CU(cudaMemcpyAsync(q.p, kmers, n * sizeof(Key<W>), cudaMemcpyHostToDevice, c->stream));
  k_lookup<W><<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(freq_table<W>(c), q.as<Key<W>>(), n, c->cfg.K, canon,
                                                                 r.as<uint32_t>());
  c->launches++;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, r.p, n * 4, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  CU(e);
  return APGK_OK;
}

template <int W>
int read_freqs_impl(apgk_ctx* c, uint64_t first, uint64_t n, uint32_t* out) {
  if (!n) return APGK_OK;
  { int rc = wait_ingest(c); if (rc) return rc; }
  struct Tmp { DevBuf b; ~Tmp() { b.release(); } } r_;   // released on every path out
  DevBuf& r = r_.b;
  CU(r.ensure(n * 4));
  constexpr int NT = 128;
  const uint64_t span = (first + n) - (first & ~15ull);
  const uint64_t threads = (span + POS_PER_THREAD - 1) / POS_PER_THREAD;
  k_read_freqs<W, NT><<<(unsigned)((threads + NT - 1) / NT), NT, 0, c->stream>>>(read_store(c), freq_table<W>(c), first, n,
                                                                               r.as<uint32_t>());
  c->launches++;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, r.p, n * 4, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  CU(e);
  return APGK_OK;
}

// ---------------------------------------------------------------- sharded counting, receiver side
// exclusive scan of a u32 array into u64[n+1] (total -> *total_out if not null)
int scan_u32(apgk_ctx* c, const uint32_t* in, uint64_t n, unsigned long long* out, unsigned long long* total_out) {
  const uint32_t nblocks = (uint32_t)((n + 1 + SCAN_BLOCK - 1) / SCAN_BLOCK);
  CU(c->blocksum.ensure(((size_t)nblocks + 1) * 8));
  k_scan_blocksum<<<nblocks, SCAN_NT, 0, c->stream>>>(in, n, c->blocksum.as<unsigned long long>());
  LAUNCHED();
  k_scan_top<<<1, SCAN_NT, 0, c->stream>>>(c->blocksum.as<unsigned long long>(), nblocks, nullptr);
  LAUNCHED();
  k_scan_apply<<<nblocks, SCAN_NT, 0, c->stream>>>(in, n, c->blocksum.as<unsigned long long>(), out);
  LAUNCHED();
  if (total_out) {
    CU(cudaMemcpyAsync(total_out, c->blocksum.as<unsigned long long>() + nblocks, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  return APGK_OK;
}

// ---------------------------------------------------------------- occurrence records
static const bool kFreqDirect = getenv("APGK_FREQ_DIRECT") != nullptr;  // whole-store read_freqs by per-window table search
static const bool kOccDirect = getenv("APGK_OCC_DIRECT") != nullptr;  // first version: lookup + slot + store straight from the sweep

struct OccScatter {
  void* elems = nullptr;
  unsigned long long* pos_tmp = nullptr;
  int pack_bits = 0;
};

// run offsets = exclusive scan of the counts, in c->occ_off; fails if a count saturated
int occ_run_offsets(apgk_ctx* c) {
  const uint64_t N = c->n_instances, D = c->n_distinct;
  CU(c->occ_off.ensure((D + 1) * 8));
  unsigned long long total = 0;
  { int rc = scan_u32(c, c->out_cnt.as<uint32_t>(), D, c->occ_off.as<unsigned long long>(), &total); if (rc) return rc; }
  if (total != N) FAIL(APGK_E_RANGE, "counts sum to %llu, instances %llu (a count saturated)", total, (unsigned long long)N);
  return APGK_OK;
}

// Phase 1 of the two-phase forms: the sweep of the reads that sends every window to its prefix bucket's region.
// The pipeline's A / B are dead after finish and reused: elements in B (32-bit remainders; unused when remainder
// and position share a word) or A (full keys), the positions on their way to their bucket in A or occ_pos.
template <int W, typename Elem>
int occ_scatter_phase(apgk_ctx* c, unsigned long long* counters, OccScatter& o) {
  const uint64_t N = c->n_instances;
  const uint32_t nb = c->nb1;
  constexpr bool U32 = sizeof(Elem) == 4;
  unsigned long long* run_off = c->occ_off.as<unsigned long long>();
  o.pack_bits = 0;
  if (U32) {
    // position bits: (q << 1 | rc) of the last base; remainder and position share one word when they fit
    int pos_bits = 1;
    while (pos_bits < 64 && (2 * c->total_bases) >> pos_bits) pos_bits++;
    if (c->geom.REM + pos_bits <= 64 && !getenv("APGK_OCC_NOPACK")) o.pack_bits = pos_bits;
    if (!o.pack_bits) CU(c->B.ensure(N * 4));
    CU(c->A.ensure(N * 8));
    o.elems = c->B.p; o.pos_tmp = c->A.as<unsigned long long>();
  } else {
    CU(c->A.ensure(N * sizeof(Elem)));
    CU(c->occ_pos.ensure(N * 8));
    o.elems = c->A.p; o.pos_tmp = c->occ_pos.as<unsigned long long>();
  }
  CU(c->occ_bstart.ensure(((size_t)nb + 1) * 8));
  CU(c->occ_bcur.ensure((size_t)nb * 8));
  k_occ_bstart<<<(nb + 1 + 255) / 256, 256, 0, c->stream>>>(c->out_off.as<unsigned long long>(), run_off, nb,
                                                         c->occ_bstart.as<unsigned long long>(),
                                                         c->occ_bcur.as<unsigned long long>());
  LAUNCHED();
  CU(cudaEventRecord(c->occ_ev[1], c->stream));
  constexpr int NT = 128;
  const uint64_t threads = (c->total_bases + POS_PER_THREAD - 1) / POS_PER_THREAD;
  k_occ_scatter<W, Elem, unsigned long long, NT><<<(unsigned)((threads + NT - 1) / NT), NT, 0, c->stream>>>(
      read_store(c), freq_table<W>(c), 0, c->total_bases, nullptr, c->occ_bcur.as<unsigned long long>(), (Elem*)o.elems, o.pos_tmp,
      o.pack_bits, N, counters);
  LAUNCHED();
  CU(cudaEventRecord(c->occ_ev[2], c->stream));
  return APGK_OK;
}

template <int W, typename Elem>
int build_occurrences_impl(apgk_ctx* c) {
  const uint64_t N = c->n_instances, D = c->n_distinct;
  c->have_occ = false; c->n_occ = 0; c->n_big_runs = 0;
  for (float& m : c->occ_ms) m = 0;
  { int rc = wait_ingest(c); if (rc) return rc; }
  for (cudaEvent_t& e : c->occ_ev) if (!e) CU(cudaEventCreate(&e));
  if (!N) {
    CU(c->occ_off.ensure((D + 1) * 8));
    CU(cudaMemsetAsync(c->occ_off.p, 0, (D + 1) * 8, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->have_occ = true;
    return APGK_OK;
  }
  CU(cudaEventRecord(c->occ_ev[0], c->stream));
  { int rc = occ_run_offsets(c); if (rc) return rc; }
  unsigned long long* run_off = c->occ_off.as<unsigned long long>();
  // the per-run cursors of the global-table path live in T, the big-run list in B once the placement is done
  CU(c->occ.ensure(N * 8));
  CU(c->T.ensure(D * 4));
  CU(c->occ_cnt.ensure(64));
  unsigned long long* counters = c->occ_cnt.as<unsigned long long>();
  CU(cudaMemsetAsync(c->T.p, 0, D * 4, c->stream));
  CU(cudaMemsetAsync(counters, 0, 32, c->stream));
  unsigned long long* occ = c->occ.as<unsigned long long>();
  if (kOccDirect) {
    constexpr int NT = 128;
    const uint64_t threads = (c->total_bases + POS_PER_THREAD - 1) / POS_PER_THREAD;
    CU(cudaEventRecord(c->occ_ev[1], c->stream));
    k_occ_fill<W, NT><<<(unsigned)((threads + NT - 1) / NT), NT, 0, c->stream>>>(read_store(c), freq_table<W>(c), run_off,
                                                                               c->T.as<uint32_t>(), occ, counters);
    LAUNCHED();
    CU(cudaEventRecord(c->occ_ev[2], c->stream));
  } else {
    OccScatter sc;
    { int rc = occ_scatter_phase<W, Elem>(c, counters, sc); if (rc) return rc; }
    k_occ_place<W, Elem, OCC_PLACE_NT, false><<<std::min<uint32_t>(c->nb1, (uint32_t)c->n_sm * 8), OCC_PLACE_NT, 0, c->stream>>>(
        freq_table<W>(c), run_off, c->occ_bstart.as<unsigned long long>(), (const Elem*)sc.elems, sc.pos_tmp, sc.pack_bits,
        c->T.as<uint32_t>(), occ, nullptr, counters);
    LAUNCHED();
  }
  CU(cudaEventRecord(c->occ_ev[3], c->stream));
  const size_t list_cap = (size_t)(N / OCC_SMALL_MAX) + 1;
  CU(c->B.ensure(list_cap * 8));
  k_occ_sort_small<<<(unsigned)((D + 127) / 128), 128, 0, c->stream>>>(run_off, D, occ, c->B.as<unsigned long long>(), counters);
  LAUNCHED();
  CU(cudaEventRecord(c->occ_ev[4], c->stream));
  k_occ_sort_big<OCC_BIG_NT><<<c->n_sm * 2, OCC_BIG_NT, 0, c->stream>>>(run_off, c->B.as<unsigned long long>(), counters, occ);
  LAUNCHED();
  CU(cudaEventRecord(c->occ_ev[5], c->stream));
  // rank directory over the start bitmap: read id of a global base position
  {
    const uint64_t words = (c->total_bases + 31) / 32;
    const uint64_t n_blocks = words / RANK_BLOCK_WORDS + 1;   // covers word index `words` as well; the bitmap is zero padded
    CU(c->rank_cnt.ensure(n_blocks * 4));
    CU(c->rank_dir.ensure((n_blocks + 1) * 8));
    k_start_blocks<<<(unsigned)((n_blocks + 255) / 256), 256, 0, c->stream>>>(c->starts.as<uint32_t>(), n_blocks,
                                                                            c->rank_cnt.as<uint32_t>());
    LAUNCHED();
    int rc = scan_u32(c, c->rank_cnt.as<uint32_t>(), n_blocks, c->rank_dir.as<unsigned long long>(), nullptr);
    if (rc) return rc;
    if (!c->empty_nb.empty()) {
      CU(c->empty_dev.ensure(c->empty_nb.size() * 8));
      CU(cudaMemcpyAsync(c->empty_dev.p, c->empty_nb.data(), c->empty_nb.size() * 8, cudaMemcpyHostToDevice, c->stream));
    }
  }
  unsigned long long h[3] = {0, 0, 0};
  CU(cudaMemcpyAsync(h, counters, 24, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  for (int i = 0; i < 5; i++) cudaEventElapsedTime(&c->occ_ms[i], c->occ_ev[i], c->occ_ev[i + 1]);
  if (kOccDirect) c->occ_ms[2] = 0;  // no placement pass in the direct form
  if (h[1] || h[2])
    FAIL(APGK_E_STATE, "occurrences: %llu windows missing from the table, %llu slots past a run (table does not match the read store)",
         h[1], h[2]);
  c->n_big_runs = h[0];
  c->n_occ = N;
  c->have_occ = true;
  return APGK_OK;
}

// Bulk form of apgk_read_freqs: the count of the canonical k-mer at EVERY base of the store (0xFFFFFFFF where the
// window leaves its read) into d_out (DEVICE, total_bases entries), by bucket scatter + per-bucket placement.
template <int W, typename Elem>
int read_freqs_bulk(apgk_ctx* c, uint32_t* d_out) {
  const uint64_t N = c->n_instances;
  { int rc = wait_ingest(c); if (rc) return rc; }
  for (cudaEvent_t& e : c->occ_ev) if (!e) CU(cudaEventCreate(&e));
  if (!c->total_bases) return APGK_OK;
  CU(cudaEventRecord(c->occ_ev[0], c->stream));
  CU(cudaMemsetAsync(d_out, 0xFF, c->total_bases * 4, c->stream));
  if (N) {
    { int rc = occ_run_offsets(c); if (rc) return rc; }
    CU(c->occ_cnt.ensure(64));
    unsigned long long* counters = c->occ_cnt.as<unsigned long long>();
    CU(cudaMemsetAsync(counters, 0, 32, c->stream));
    OccScatter sc;
    { int rc = occ_scatter_phase<W, Elem>(c, counters, sc); if (rc) return rc; }
    k_occ_place<W, Elem, OCC_PLACE_NT, true><<<std::min<uint32_t>(c->nb1, (uint32_t)c->n_sm * 8), OCC_PLACE_NT, 0, c->stream>>>(
        freq_table<W>(c), c->occ_off.as<unsigned long long>(), c->occ_bstart.as<unsigned long long>(), (const Elem*)sc.elems,
        sc.pos_tmp, sc.pack_bits, nullptr, nullptr, d_out, counters);
    LAUNCHED();
    CU(cudaEventRecord(c->occ_ev[3], c->stream));
    unsigned long long h[3] = {0, 0, 0};
    CU(cudaMemcpyAsync(h, counters, 24, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    cudaEventElapsedTime(&c->freq_ms[0], c->occ_ev[0], c->occ_ev[1]);
    cudaEventElapsedTime(&c->freq_ms[1], c->occ_ev[1], c->occ_ev[2]);
    cudaEventElapsedTime(&c->freq_ms[2], c->occ_ev[2], c->occ_ev[3]);
    if (h[1] || h[2])
      FAIL(APGK_E_STATE, "read_freqs: %llu windows missing from the table, %llu slots past a bucket (table does not match the read store)",
           h[1], h[2]);
  } else {
    CU(cudaStreamSynchronize(c->stream));
  }
  return APGK_OK;
}

int read_freqs_bulk_dispatch(apgk_ctx* c, uint32_t* d_out) {
  switch (c->W) {
    case 1: return c->geom.REM <= 32 ? read_freqs_bulk<1, uint32_t>(c, d_out) : read_freqs_bulk<1, Key<1>>(c, d_out);
    case 2: return read_freqs_bulk<2, Key<2>>(c, d_out);
    case 3: return read_freqs_bulk<3, Key<3>>(c, d_out);
  }
  return APGK_E_ARG;
}

int occurrences_copy_impl(apgk_ctx* c, uint64_t first, uint64_t n_kmers, uint64_t* run_off_out, uint32_t* read_id_out,
                          int32_t* pos_out) {
  std::vector<unsigned long long> ends(2, 0);
  const unsigned long long* off = c->occ_off.as<unsigned long long>();
  CU(cudaMemcpyAsync(&ends[0], off + first, 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(&ends[1], off + first + n_kmers, 8, cudaMemcpyDeviceToHost, c->stream));
  if (run_off_out)
    CU(cudaMemcpyAsync(run_off_out, off + first, (n_kmers + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  if (!read_id_out && !pos_out) return APGK_OK;
  const uint64_t o0 = ends[0], n = ends[1] - ends[0];
  const uint64_t CH = 1ull << 26;  // occurrences translated per step (768 MB of device scratch at most)
  CU(c->occ_tmp.ensure(std::min(n, CH) * 8 + 8));
  uint32_t* d_id = c->occ_tmp.as<uint32_t>();
  for (uint64_t done = 0; done < n; done += CH) {
    const uint64_t m = std::min(CH, n - done);
    int32_t* d_pos = (int32_t*)(d_id + m);
    k_occ_translate<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(
        c->occ.as<unsigned long long>() + o0 + done, m, c->starts.as<uint32_t>(), c->rank_dir.as<unsigned long long>(),
        c->empty_dev.as<unsigned long long>(), (uint32_t)c->empty_nb.size(), d_id, d_pos);
    LAUNCHED();
    if (read_id_out) CU(cudaMemcpyAsync(read_id_out + done, d_id, m * 4, cudaMemcpyDeviceToHost, c->stream));
    if (pos_out) CU(cudaMemcpyAsync(pos_out + done, d_pos, m * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  return APGK_OK;
}

// split bits actually used for a request (same on every rank: it depends on the geometry only)
int effective_split_bits(const apgk_ctx* c, int d2) {
  d2 = std::max(0, std::min(d2, 5));
  d2 = std::min(d2, std::max(0, c->geom.REM - 1));
  while (d2 > 0 && c->geom.D0 + c->geom.D1 + d2 > 27) d2--;
  return d2;
}

template <int W, typename ElemB>
int sub_sizes_typed(apgk_ctx* c, int d2) {
  const uint32_t nb = c->nb1;
  CU(c->sub_sizes.ensure(((size_t)nb << d2) * 4 + 16));
  if (!c->part_n) { CU(cudaMemsetAsync(c->sub_sizes.p, 0, ((size_t)nb << d2) * 4, c->stream)); }
  else {
    k_sub_hist<ElemB, 256><<<c->n_sm * 8, 256, 0, c->stream>>>(c->B.as<ElemB>(), c->bofs.as<unsigned long long>(),
                                                               c->segtot.as<unsigned long long>(), nb, d2, c->geom.REM - d2,
                                                               c->sub_sizes.as<uint32_t>());
    LAUNCHED();
  }
  CU(cudaStreamSynchronize(c->stream));
  return APGK_OK;
}

template <int W, typename ElemB>
int count_pieces_typed(apgk_ctx* c, const void* const* bases_host, bool peer, uint32_t n_src, const uint32_t* d_sizes_all,
                       const uint64_t* seg_off_host, uint32_t lo, uint32_t hi, int d2, const uint32_t* d_sub) {
  const uint32_t nb = c->nb1;
  // split bits: every merged bucket is cut into 2^d2 sub-buckets by the leading remainder bits
  d2 = effective_split_bits(c, d2);
  const uint32_t nbf = nb << d2;
  stages_reset(c);
  stage_begin(c, ST_TOTAL);
  stage_begin(c, ST_OWNER);
  CU(c->segtot.ensure((size_t)nbf * 8));
  CU(c->nd.ensure(((size_t)nbf + 1) * 4));
  CU(c->bofs.ensure(((size_t)nbf + 1) * 8));
  CU(c->out_off_local.ensure(((size_t)nbf + 1) * 8));
  CU(c->out_off.ensure(((size_t)nbf + 1) * 8));
  CU(c->stats.ensure(64));
  CU(c->misc.ensure(64));
  CU(c->bstart64.ensure(std::max<size_t>(((size_t)(1u << c->geom.D0) + 1) * 8, (size_t)n_src * 8)));
  CU(cudaMemsetAsync(c->misc.p, 0, 64, c->stream));
  // merged (coarse) bucket sizes -> nd, their offsets -> out_off_local (both are free until the counting starts)
  k_merge_sizes<<<(nb + 255) / 256, 256, 0, c->stream>>>(d_sizes_all, n_src, nb, lo, hi, c->nd.as<uint32_t>(),
                                                       c->misc.as<unsigned int>());
  LAUNCHED();
  unsigned long long Nr = 0;
  { int rc = scan_u32(c, c->nd.as<uint32_t>(), nb, c->out_off_local.as<unsigned long long>(), &Nr); if (rc) return rc; }
  unsigned int ovf = 0;
  CU(cudaMemcpyAsync(&ovf, c->misc.p, 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  if (ovf) FAIL(APGK_E_RANGE, "a merged bucket holds 2^32 or more k-mers");
  // offset of every piece inside its source's segment
  CU(c->piece_off.ensure((size_t)n_src * ((size_t)nb + 1) * 8));
  CU(c->piece_tmp.ensure((size_t)nb * 4));
  for (uint32_t s = 0; s < n_src; s++) {
    k_mask_sizes<<<(nb + 255) / 256, 256, 0, c->stream>>>(d_sizes_all + (size_t)s * nb, nb, lo, hi, c->piece_tmp.as<uint32_t>());
    LAUNCHED();
    int rc = scan_u32(c, c->piece_tmp.as<uint32_t>(), nb, c->piece_off.as<unsigned long long>() + (size_t)s * (nb + 1), nullptr);
    if (rc) return rc;
  }
  CU(c->piece_ptrs.ensure((size_t)n_src * 8));
  CU(cudaMemcpyAsync(c->piece_ptrs.p, bases_host, (size_t)n_src * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->bstart64.p, seg_off_host, (size_t)n_src * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));  // the host arrays may die
  // the gathered shard: over the dead send buffer B after an all-to-all; a second buffer when the peers
  // (and this rank itself) are still reading B
  DevBuf& dst = peer ? c->C2 : c->B;
  CU(dst.ensure(std::max<size_t>(Nr, 1) * sizeof(ElemB) + 16));
  CU(c->A.ensure(std::max<size_t>(Nr, 1) * sizeof(Key<W>)));
  CU(cudaMemsetAsync(c->segtot.p, 0, (size_t)nbf * 8, c->stream));
  CU(cudaMemsetAsync(c->bofs.p, 0, ((size_t)nbf + 1) * 8, c->stream));
  if (Nr && hi > lo) {
    const uint32_t grid = std::min<uint32_t>((hi - lo + 7) / 8, (uint32_t)c->n_sm * 8);  // one warp per bucket
    // digit = the d2 bits just below the prefix: remainder bits [REM - d2, REM)
    GatherArgs<ElemB> ga{};
    ga.src_base = (const ElemB* const*)c->piece_ptrs.p; ga.seg_off = c->bstart64.as<unsigned long long>();
    ga.piece_off = c->piece_off.as<unsigned long long>(); ga.sizes_all = d_sizes_all;
    ga.bofs_coarse = c->out_off_local.as<unsigned long long>(); ga.coarse_base = 0;
    ga.n_src = n_src; ga.nb = nb; ga.lo = lo; ga.hi = hi; ga.d2 = d2; ga.digit_pos = c->geom.REM - d2;
    ga.out = (ElemB*)dst.p; ga.bsize_fine = c->segtot.as<unsigned long long>(); ga.bofs_fine = c->bofs.as<unsigned long long>();
    ga.sub_sizes = d_sub; ga.sub_ptrs = nullptr;
    k_gather_split<ElemB, 256><<<grid, 256, 0, c->stream>>>(ga);
    LAUNCHED();
  }
  stage_end(c, ST_OWNER);
  // from here on the context describes the finer geometry: P + d2 prefix bits
  c->geom.D1 += d2; c->geom.REM -= d2;
  c->nb1 = nbf;
  c->part_ready = false;   // the partition's geometry is gone: a failed count cannot be retried on it
  c->n_instances = Nr;
  c->n_big = 0;
  uint64_t n_prev = 0;
  CU(c->spec_ovf.ensure(((size_t)Nr / SPEC_DENSE + 16) * 8));
  CU(cudaMemsetAsync(c->spec_ovf.p, 0, 8, c->stream));
  CU(cudaMemsetAsync(c->spec_dense.p, 0, (size_t)SPEC_DENSE * 8, c->stream));
  CU(cudaMemsetAsync(c->out_off.p, 0, ((size_t)nbf + 1) * 8, c->stream));
  c->count_src = dst.p;
  c->bucket_lo = lo << d2; c->bucket_hi = hi << d2;
  CU(c->res.ensure(RES_WORDS * 8));
  if (Nr) { int rc = count_buckets<W, ElemB>(c, Nr, Nr, n_prev, c->A.as<Key<W>>(), false); if (rc) return rc; }
  c->n_distinct = n_prev;
  c->have_table = (c->cfg.flags & APGK_WANT_COUNTS) != 0;
  stage_end(c, ST_TOTAL);
  c->n_deferred = 0;
  if (c->deferred.p && Nr) CU(cudaMemcpyAsync(&c->n_deferred, c->deferred.p, 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  stages_collect(c);
  c->part_ready = false;
  c->spec_loaded = false;
  c->finished = true;
  return APGK_OK;
}

template <int W>
int count_pieces_impl(apgk_ctx* c, const void* const* bases_host, bool peer, uint32_t n_src, const uint32_t* d_sizes_all,
                      const uint64_t* seg_off_host, uint64_t lo, uint64_t hi, int d2, const uint32_t* d_sub) {
  if (!c->part_ready) FAIL(APGK_E_STATE, "apgk_count_pieces needs a preceding apgk_partition on this context");
  if (n_src == 0 || n_src > 1024 || lo > hi || hi > c->nb1) FAIL(APGK_E_ARG, "apgk_count_pieces: bad source count or bucket range");
  if constexpr (W == 1) {
    if (c->elem_bytes == 4) return count_pieces_typed<W, uint32_t>(c, bases_host, peer, n_src, d_sizes_all, seg_off_host, (uint32_t)lo, (uint32_t)hi, d2, d_sub);
  }
  return count_pieces_typed<W, Key<W>>(c, bases_host, peer, n_src, d_sizes_all, seg_off_host, (uint32_t)lo, (uint32_t)hi, d2, d_sub);
}

// ---------------------------------------------------------------- owner partition (multi-GPU shuffle, sender side)
template <int W>
int owner_plan_impl(apgk_ctx* c, uint32_t n_ranks, uint64_t* counts_out) {
  { int rc = wait_ingest(c); if (rc) return rc; }
  DigitSpec ds{DIGIT_OWNER, 0, 0, 0, n_ranks};
  const DigitFn<DIGIT_OWNER> dg = make_digit_fn<DIGIT_OWNER>(ds);
  const uint32_t tile0 = (uint32_t)Geo<W>::NT0 * POS_PER_THREAD;
  HostPlan& hp = c->owner_plan;
  std::vector<uint64_t> one{c->total_bases};
  build_plan(hp, one, tile0, (int)n_ranks);
  c->owner_counts.assign(n_ranks, 0);
  c->owner_ranks = n_ranks; c->owner_tiles = hp.lp.n_tiles;
  if (hp.lp.n_tiles) {
    // the owner plan keeps its own device copy: apgk_owner_scatter runs later
    const size_t S1 = hp.seg_tile0.size();
    CU(c->owner_plan_dev.ensure(S1 * 16 + 64));
    unsigned char* d = c->owner_plan_dev.as<unsigned char>();
    CU(cudaMemcpyAsync(d, hp.seg_start.data(), S1 * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d + S1 * 8, hp.seg_tile0.data(), S1 * 4, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d + S1 * 12, hp.seg_chunk0.data(), S1 * 4, cudaMemcpyHostToDevice, c->stream));
    hp.lp.seg_start = (const uint64_t*)d;
    hp.lp.seg_tile0 = (const uint32_t*)(d + S1 * 8);
    hp.lp.seg_chunk0 = (const uint32_t*)(d + S1 * 12);
    CU(c->chunksum.ensure((size_t)hp.lp.n_chunks * n_ranks * 4));
    stage_begin(c, ST_OWNER);
    k_hist_reads<W, Geo<W>::NT0, DIGIT_OWNER><<<hp.lp.n_chunks, Geo<W>::NT0, n_ranks * 4, c->stream>>>(
        read_store(c), dg, hp.lp, 0, c->chunksum.as<uint32_t>());
    LAUNCHED();
    { int rc = column_scan(c, hp, 0, nullptr); if (rc) return rc; }
    CU(cudaMemcpyAsync(c->owner_counts.data(), c->segtot.p, (size_t)n_ranks * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  for (uint32_t r = 0; r < n_ranks; r++) {
    if (c->owner_counts[r] >= (1ull << 32)) FAIL(APGK_E_RANGE, "more than 2^32 k-mers for one owner in one call");
    counts_out[r] = c->owner_counts[r];
  }
  return APGK_OK;
}

template <int W>
int owner_scatter_impl(apgk_ctx* c, uint64_t* d_out) {
  const uint32_t n_ranks = c->owner_ranks;
  if (!c->owner_tiles) return APGK_OK;
  DigitSpec ds{DIGIT_OWNER, 0, 0, 0, n_ranks};
  const DigitFn<DIGIT_OWNER> dg = make_digit_fn<DIGIT_OWNER>(ds);
  std::vector<uint64_t> bstart(n_ranks + 1, 0);
  for (uint32_t r = 0; r < n_ranks; r++) bstart[r + 1] = bstart[r] + c->owner_counts[r];
  CU(c->bstart64.ensure(((size_t)n_ranks + 1) * 8));
  CU(cudaMemcpyAsync(c->bstart64.p, bstart.data(), ((size_t)n_ranks + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  auto kern = k_scatter_reads<W, Geo<W>::NTS, DIGIT_OWNER, false, Geo<W>::NPOS>;
  const size_t sm = scatter_smem_bytes<Key<W>>((uint32_t)Geo<W>::NT0 * POS_PER_THREAD, (int)n_ranks);
  { int rc = set_smem(c, kern, sm); if (rc) return rc; }
  kern<<<c->owner_plan.lp.n_chunks, Geo<W>::NTS, sm, c->stream>>>(read_store(c), dg, c->owner_plan.lp,
                                                                  c->chunksum.as<uint32_t>(), c->bstart64.as<uint64_t>(),
                                                                  (Key<W>*)d_out);
  LAUNCHED();
  stage_end(c, ST_OWNER);
  CU(cudaStreamSynchronize(c->stream));
  return APGK_OK;
}

}  // namespace

namespace {
template <int W>
static void host_table_find(int K, const uint64_t* sorted, uint64_t n, int P, const uint64_t* q, uint64_t nq, uint64_t* out) {
  const int TB = std::max(2 * K, P), pad = TB - 2 * K, REM = TB - P;
  std::vector<unsigned long long> index(((size_t)1 << P) + 1, 0);
  const Key<W>* keys = (const Key<W>*)sorted;
  for (uint64_t i = 0; i < n; i++) index[digit_of(keys[i], REM, P, pad) + 1]++;
  for (size_t b = 0; b < ((size_t)1 << P); b++) index[b + 1] += index[b];
  FreqTable<W> t;
  t.keys = keys; t.counts = nullptr; t.index = index.data(); t.nb = 1u << P;
  t.prefix_pos = REM; t.prefix_len = P; t.pad = pad; t.D1 = 0;
  for (uint64_t i = 0; i < nq; i++) out[i] = table_find_index(t, ((const Key<W>*)q)[i]);
}

template <int W>
static void host_extract(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, int K, uint64_t* kmers_out,
                         uint8_t* valid_out) {
  const uint64_t b0 = off[0], total = off[n_reads] - b0;
  // build the store exactly as the device sees it: bases from position 0, zero padded
  std::vector<uint32_t> bases((total + 15) / 16 + 2 * W + 8, 0), starts((total + 31) / 32 + 16, 0);
  for (uint64_t q = 0; q < total; q++) {
    const uint64_t s = b0 + q;
    const uint32_t b = (packed[s >> 2] >> ((s & 3) * 2)) & 3u;
    bases[q >> 4] |= b << ((q & 15) * 2);
  }
  for (uint64_t r = 0; r < n_reads; r++) { const uint64_t q = off[r] - b0; starts[q >> 5] |= 1u << (q & 31); }
  for (uint64_t p = 0; p < total; p += 16) {
    const uint32_t valid = window_valid_mask16(starts.data(), p, K, total);
    Window16<W> win;
    load_window16<W>(bases.data(), p, K, win);
    extract16<W>(win, K, [&](int j, const Key<W>& c, bool) {
      if (p + j < total) {
        valid_out[p + j] = (valid >> j) & 1u;
        for (int i = 0; i < W; i++) kmers_out[(p + j) * W + i] = c.w[i];
      }
    });
  }
}

}  // namespace

#include "group.cuh"

// ================================================================= C ABI
extern "C" {

int apgk_words_per_kmer(int K) { return words_for(K); }

int apgk_create(const apgk_config* cfg, apgk_ctx** out) {
  if (!cfg || !out) return APGK_E_ARG;
  *out = nullptr;
  if (cfg->K < 1 || cfg->K > APGK_MAX_K) return APGK_E_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return APGK_E_CUDA;  // no CPU fallback
  if (cfg->device < 0 || cfg->device >= ndev) return APGK_E_ARG;
  if (cudaSetDevice(cfg->device) != cudaSuccess) return APGK_E_CUDA;
  apgk_ctx* c = new apgk_ctx();
  c->cfg = *cfg;
  c->cfg.flags |= APGK_WANT_SPECTRUM;
  c->W = words_for(cfg->K);
  c->device = cfg->device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) { delete c; return APGK_E_CUDA; }
  c->n_sm = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return APGK_E_CUDA; }
  stages_reset(c);
  if (cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { apgk_destroy(c); return APGK_E_CUDA; }
  cudaEventCreateWithFlags(&c->ev_main, cudaEventDisableTiming);
  if (cfg->reserve_bases && ensure_store(c, cfg->reserve_bases) != APGK_OK) {
    apgk_destroy(c);
    return APGK_E_NOMEM;
  }
  *out = c;
  return APGK_OK;
}

void apgk_destroy(apgk_ctx* c) {
  if (!c) return;
  if (c->group) group_detach(c->group, c);   // whichever of the two is destroyed first, nothing dangles
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  DevBuf* all[] = {&c->tot0_dev, &c->res, &c->bases, &c->starts, &c->staging, &c->off_dev, &c->A, &c->B, &c->T, &c->chunksum, &c->chunksum0, &c->plan0, &c->out_off_local,
                   &c->segtot, &c->bstart32, &c->bofs, &c->plan, &c->bstart64, &c->nd, &c->out_off, &c->blocksum,
                   &c->big_list, &c->stats, &c->scratch, &c->stacks, &c->spec_dense, &c->spec_ovf, &c->misc, &c->deferred,
                   &c->out_keys, &c->out_cnt, &c->owner_plan_dev, &c->piece_off, &c->piece_tmp, &c->piece_ptrs, &c->C2, &c->sub_sizes, &c->TK,
                   &c->occ, &c->occ_pos, &c->occ_off, &c->occ_cnt, &c->occ_bstart, &c->occ_bcur, &c->rank_cnt, &c->rank_dir, &c->empty_dev,
                   &c->occ_tmp};
  for (DevBuf* b : all) b->release();
  for (cudaEvent_t e : c->occ_ev) if (e) cudaEventDestroy(e);
  for (auto& iv : c->ivs) { cudaEventDestroy(iv.e0); cudaEventDestroy(iv.e1); }
  if (c->res_host) cudaFreeHost(c->res_host);
  if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
  for (cudaEvent_t e : c->slice_ev) cudaEventDestroy(e);
  if (c->ev_main) cudaEventDestroy(c->ev_main);
  cudaStreamDestroy(c->stream);
  delete c;
}

const char* apgk_last_error(const apgk_ctx* c) { return c ? c->err.c_str() : "null context"; }

int apgk_reset(apgk_ctx* c) {
  if (!c) return APGK_E_ARG;
  c->gen++;
  CU(cudaSetDevice(c->device));
  { int rc = wait_ingest(c); if (rc) return rc; }
  if (c->total_bases) {
    CU(cudaMemsetAsync(c->bases.p, 0, std::min(c->bases.cap, (size_t)((c->total_bases + 31) / 32) * 8 + 256), c->stream));
    CU(cudaMemsetAsync(c->starts.p, 0, std::min(c->starts.cap, (size_t)((c->total_bases + 31) / 32) * 4 + 256), c->stream));
  }
  c->total_bases = 0; c->n_reads = 0; c->n_windows = 0;
  c->empty_nb.clear();
  invalidate_results(c);
  return APGK_OK;
}

int apgk_add_reads(apgk_ctx* c, const uint8_t* packed, const uint64_t* off, uint64_t n_reads) {
  if (!c || (!packed && n_reads) || (!off && n_reads)) return APGK_E_ARG;
  c->gen++;
  if (!n_reads) return APGK_OK;
  CU(cudaSetDevice(c->device));
  { int rc = wait_ingest(c); if (rc) return rc; }
  for (uint64_t r = 0; r < n_reads; r++)
    if (off[r + 1] < off[r]) FAIL(APGK_E_ARG, "read offsets must be non-decreasing (read %llu)", (unsigned long long)r);
  const uint64_t nb = off[n_reads] - off[0];
  const uint64_t dst0 = c->total_bases;
  int rc = append_bases(c, packed, off[0], nb);
  if (rc) return rc;
  if (nb) {
    CU(c->off_dev.ensure(n_reads * 8));
    CU(cudaMemcpyAsync(c->off_dev.p, off, n_reads * 8, cudaMemcpyHostToDevice, c->stream));
    k_mark_starts<<<(unsigned)((n_reads + 255) / 256), 256, 0, c->stream>>>(c->off_dev.as<uint64_t>(), n_reads, off[0],
                                                                           dst0, c->starts.as<uint32_t>());
    LAUNCHED();
  }
  CU(cudaStreamSynchronize(c->stream));  // inputs are only borrowed for the duration of the call
  for (uint64_t r = 0; r < n_reads; r++) {  // reads without bases own no start bit: remember where they sit (occurrence read ids)
    const uint64_t len = off[r + 1] - off[r];
    if (len == 0) c->empty_nb.push_back(c->n_reads + r - c->empty_nb.size());
    if (len >= (uint64_t)c->cfg.K) c->n_windows += len - (uint64_t)c->cfg.K + 1;
  }
  c->total_bases += nb; c->n_reads += n_reads;
  invalidate_results(c);
  return APGK_OK;
}

int apgk_add_reads_uniform(apgk_ctx* c, const uint8_t* packed, uint64_t first_base, uint64_t n_reads, uint32_t read_len) {
  if (!c || (!packed && n_reads)) return APGK_E_ARG;
  c->gen++;
  if (!n_reads || !read_len) return APGK_OK;
  CU(cudaSetDevice(c->device));
  const uint64_t nb = n_reads * (uint64_t)read_len;
  const uint64_t dst0 = c->total_bases;
  const bool aligned = ((2 * dst0) & 7) == 0 && ((2 * first_base) & 7) == 0 && ((2 * nb) & 7) == 0;
  if ((c->cfg.flags & APGK_ASYNC_INGEST) && aligned && c->n_slices == 0) {
    // streamed ingest: the copy goes out in slices on its own stream; finish / partition follow it slice by slice
    { int rc = ensure_store(c, dst0 + nb); if (rc) return rc; }
    const size_t nbytes = (size_t)(nb / 4);
    const size_t n_sl = std::max<size_t>(1, std::min<size_t>(16, nbytes >> 24));  // slices of >= 16 MB
    while (c->slice_ev.size() < n_sl) {
      cudaEvent_t e;
      CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      c->slice_ev.push_back(e);
    }
    c->slice_end.assign(n_sl, 0);
    CU(cudaEventRecord(c->ev_main, c->stream));            // the store's memsets / earlier kernels come first
    CU(cudaStreamWaitEvent(c->copy_stream, c->ev_main, 0));
    const size_t per = ((nbytes / n_sl) + 4095) & ~(size_t)4095;
    uint8_t* dst = c->bases.as<uint8_t>() + (2 * dst0 >> 3);
    const uint8_t* src = packed + (2 * first_base >> 3);
    size_t done = 0;
    for (size_t i = 0; i < n_sl; i++) {
      const size_t len = (i + 1 == n_sl) ? nbytes - done : std::min(per, nbytes - done);
      if (len) CU(cudaMemcpyAsync(dst + done, src + done, len, cudaMemcpyHostToDevice, c->copy_stream));
      done += len;
      CU(cudaEventRecord(c->slice_ev[i], c->copy_stream));
      c->slice_end[i] = dst0 + (uint64_t)done * 4;
    }
    k_mark_starts_uniform<<<(unsigned)((n_reads + 255) / 256), 256, 0, c->stream>>>(n_reads, read_len, dst0,
                                                                                   c->starts.as<uint32_t>());
    LAUNCHED();
    c->total_bases += nb; c->n_reads += n_reads;
    if (read_len >= (uint32_t)c->cfg.K) c->n_windows += n_reads * (uint64_t)(read_len - (uint32_t)c->cfg.K + 1);
    invalidate_results(c);
    c->n_slices = n_sl;
    return APGK_OK;
  }
  { int rc = wait_ingest(c); if (rc) return rc; }
  int rc = append_bases(c, packed, first_base, nb);
  if (rc) return rc;
  k_mark_starts_uniform<<<(unsigned)((n_reads + 255) / 256), 256, 0, c->stream>>>(n_reads, read_len, dst0,
                                                                                 c->starts.as<uint32_t>());
  LAUNCHED();
  CU(cudaStreamSynchronize(c->stream));
  c->total_bases += nb; c->n_reads += n_reads;
  if (read_len >= (uint32_t)c->cfg.K) c->n_windows += n_reads * (uint64_t)(read_len - (uint32_t)c->cfg.K + 1);
  invalidate_results(c);
  return APGK_OK;
}

int apgk_synth_reads(apgk_ctx* c, const apgk_synth_params* p, uint64_t r0, uint64_t n_reads) {
  if (!c || !p) return APGK_E_ARG;
  c->gen++;
  if (!n_reads) return APGK_OK;
  if (p->read_len == 0 || p->genome_len < p->read_len) FAIL(APGK_E_ARG, "genome shorter than a read");
  if (c->total_bases % 16) FAIL(APGK_E_STATE, "apgk_synth_reads needs the store to hold a multiple of 16 bases");
  CU(cudaSetDevice(c->device));
  { int rc = wait_ingest(c); if (rc) return rc; }
  const uint64_t nb = n_reads * (uint64_t)p->read_len;
  int rc = ensure_store(c, c->total_bases + nb);
  if (rc) return rc;
  SynthParams sp{p->genome_len, p->seed_g, p->seed_p, p->seed_q, p->seed_r, p->seed_e, p->read_len, p->err_per_200};
  const uint64_t nwords = (nb + 15) / 16;
  k_synth<<<(unsigned)((nwords + 255) / 256), 256, 0, c->stream>>>(sp, r0, n_reads, c->total_bases, c->bases.as<uint32_t>());
  LAUNCHED();
  k_mark_starts_uniform<<<(unsigned)((n_reads + 255) / 256), 256, 0, c->stream>>>(n_reads, p->read_len, c->total_bases,
                                                                                 c->starts.as<uint32_t>());
  LAUNCHED();
  CU(cudaStreamSynchronize(c->stream));
  c->total_bases += nb; c->n_reads += n_reads;
  if (p->read_len >= (uint32_t)c->cfg.K) c->n_windows += n_reads * (uint64_t)(p->read_len - (uint32_t)c->cfg.K + 1);
  invalidate_results(c);
  return APGK_OK;
}

int apgk_export_reads(apgk_ctx* c, uint8_t* out) {
  if (!c || !out) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  { int rc = wait_ingest(c); if (rc) return rc; }
  if (c->total_bases) {
    CU(cudaMemcpyAsync(out, c->bases.p, ((c->total_bases + 31) / 32) * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  return APGK_OK;
}

int apgk_read_store_info(const apgk_ctx* c, uint64_t* total_bases, uint64_t* n_reads) {
  if (!c) return APGK_E_ARG;
  if (total_bases) *total_bases = c->total_bases;
  if (n_reads) *n_reads = c->n_reads;
  return APGK_OK;
}

int apgk_finish(apgk_ctx* c) {
  if (!c) return APGK_E_ARG;
  c->gen++;
  CU(cudaSetDevice(c->device));
  int rc = APGK_E_ARG;
  switch (c->W) {
    case 1: rc = finish_impl<1>(c, nullptr, 0); break;
    case 2: rc = finish_impl<2>(c, nullptr, 0); break;
    case 3: rc = finish_impl<3>(c, nullptr, 0); break;
  }
  if (rc == APGK_OK) c->table_from_reads = true;
  return rc;
}

int apgk_finish_keys_device(apgk_ctx* c, const uint64_t* d_keys, uint64_t n) {
  if (!c || (!d_keys && n)) return APGK_E_ARG;
  c->gen++;
  CU(cudaSetDevice(c->device));
  {  // the level-0 scatter writes c->A: keys handed in through apgk_key_buffer would be read and overwritten at once
    const unsigned char* k0 = (const unsigned char*)d_keys;
    const unsigned char* a0 = (const unsigned char*)c->A.p;
    if (n && a0 && k0 < a0 + c->A.cap && a0 < k0 + n * (size_t)c->W * 8)
      FAIL(APGK_E_ARG, "apgk_finish_keys_device: d_keys overlaps the library's own key buffer (apgk_key_buffer): it is the "
                       "scatter's destination -- receive into a buffer of your own");
  }
  switch (c->W) {
    case 1: return finish_impl<1>(c, (const Key<1>*)d_keys, n);
    case 2: return finish_impl<2>(c, (const Key<2>*)d_keys, n);
    case 3: return finish_impl<3>(c, (const Key<3>*)d_keys, n);
  }
  return APGK_E_ARG;
}

int apgk_window_upper(const apgk_ctx* c, uint64_t* upper) {
  if (!c || !upper) return APGK_E_ARG;
  *upper = window_upper(c);
  return APGK_OK;
}

int apgk_choose_prefix_bits(apgk_ctx* c, uint64_t upper, int32_t* prefix_bits) {
  if (!c || !prefix_bits) return APGK_E_ARG;
  switch (c->W) {
    case 1: select_geometry<1>(c, upper, 0); break;
    case 2: select_geometry<2>(c, upper, 0); break;
    case 3: select_geometry<3>(c, upper, 0); break;
    default: return APGK_E_ARG;
  }
  *prefix_bits = c->geom.D0 + c->geom.D1;
  return APGK_OK;
}

int apgk_partition(apgk_ctx* c, int32_t prefix_bits) {
  if (!c || prefix_bits < 0 || prefix_bits > 24) return APGK_E_ARG;
  c->gen++;
  CU(cudaSetDevice(c->device));
  switch (c->W) {
    case 1: return finish_impl<1>(c, nullptr, 0, RUN_PARTITION, prefix_bits);
    case 2: return finish_impl<2>(c, nullptr, 0, RUN_PARTITION, prefix_bits);
    case 3: return finish_impl<3>(c, nullptr, 0, RUN_PARTITION, prefix_bits);
  }
  return APGK_E_ARG;
}

int apgk_partition_range(apgk_ctx* c, int32_t prefix_bits, int32_t d0_lo, int32_t d0_hi) {
  if (!c || prefix_bits < 2 || prefix_bits > 24 || d0_lo < 0 || d0_hi < d0_lo) return APGK_E_ARG;
  c->force_d0_lo = d0_lo; c->force_d0_hi = d0_hi;
  const int rc = apgk_partition(c, prefix_bits);
  c->force_d0_lo = c->force_d0_hi = -1;
  return rc;
}
int apgk_level0_totals(apgk_ctx* c, uint64_t* totals_out, uint32_t cap, uint32_t* n_level0, uint64_t* round_capacity) {
  if (!c) return APGK_E_ARG;
  if (c->tot0_host.empty()) FAIL(APGK_E_STATE, "no level-0 histogram yet: call apgk_partition (it may fail with APGK_E_RANGE) first");
  if (n_level0) *n_level0 = (uint32_t)c->tot0_host.size();
  if (round_capacity) *round_capacity = c->last_cap_keys;
  if (totals_out) {
    if (cap < c->tot0_host.size()) FAIL(APGK_E_ARG, "totals_out holds %u entries, %zu needed", cap, c->tot0_host.size());
    memcpy(totals_out, c->tot0_host.data(), c->tot0_host.size() * 8);
  }
  return APGK_OK;
}
int apgk_partition_info(apgk_ctx* c, const uint64_t** d_bucket_sizes, uint64_t* n_buckets, void** d_elems,
                        uint32_t* elem_bytes, uint64_t* n_elems) {
  if (!c) return APGK_E_ARG;
  if (!c->part_ready) FAIL(APGK_E_STATE, "apgk_partition has not run");
  if (d_bucket_sizes) *d_bucket_sizes = c->segtot.as<uint64_t>();
  if (n_buckets) *n_buckets = c->nb1;
  if (d_elems) *d_elems = c->part_n ? c->B.p : nullptr;
  if (elem_bytes) *elem_bytes = c->elem_bytes;
  if (n_elems) *n_elems = c->part_n;
  return APGK_OK;
}

int apgk_partition_subsizes(apgk_ctx* c, int32_t split_bits, int32_t* effective_bits, const uint32_t** d_sub_sizes) {
  if (!c || !effective_bits || !d_sub_sizes) return APGK_E_ARG;
  if (!c->part_ready) FAIL(APGK_E_STATE, "apgk_partition has not run");
  CU(cudaSetDevice(c->device));
  const int d2 = effective_split_bits(c, split_bits);
  *effective_bits = d2;
  int rc = APGK_E_ARG;
  switch (c->W) {
    case 1: rc = c->elem_bytes == 4 ? sub_sizes_typed<1, uint32_t>(c, d2) : sub_sizes_typed<1, Key<1>>(c, d2); break;
    case 2: rc = sub_sizes_typed<2, Key<2>>(c, d2); break;
    case 3: rc = sub_sizes_typed<3, Key<3>>(c, d2); break;
  }
  *d_sub_sizes = c->sub_sizes.as<uint32_t>();
  return rc;
}

int apgk_count_pieces(apgk_ctx* c, const void* d_recv, uint32_t n_src, const uint32_t* d_sizes_all,
                      const uint64_t* seg_off, uint64_t bucket_lo, uint64_t bucket_hi, int32_t split_bits) {
  if (!c || !d_sizes_all || !seg_off || n_src == 0 || n_src > 1024) return APGK_E_ARG;
  c->gen++;
  CU(cudaSetDevice(c->device));
  std::vector<const void*> bases(n_src, d_recv);
  switch (c->W) {
    case 1: return count_pieces_impl<1>(c, bases.data(), false, n_src, d_sizes_all, seg_off, bucket_lo, bucket_hi, split_bits, nullptr);
    case 2: return count_pieces_impl<2>(c, bases.data(), false, n_src, d_sizes_all, seg_off, bucket_lo, bucket_hi, split_bits, nullptr);
    case 3: return count_pieces_impl<3>(c, bases.data(), false, n_src, d_sizes_all, seg_off, bucket_lo, bucket_hi, split_bits, nullptr);
  }
  return APGK_E_ARG;
}

int apgk_partition_export(apgk_ctx* c, uint8_t handle_out[64]) {
  if (!c || !handle_out) return APGK_E_ARG;
  if (!c->part_ready) FAIL(APGK_E_STATE, "apgk_partition has not run");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  CU(cudaSetDevice(c->device));
  CU(c->B.ensure(16));  // an empty partition still exports a valid buffer
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, c->B.p));
  memcpy(handle_out, &h, 64);
  return APGK_OK;
}

int apgk_peer_open(apgk_ctx* c, const uint8_t handle[64], void** d_ptr) {
  if (!c || !handle || !d_ptr) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  CU(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return APGK_OK;
}

int apgk_peer_close(apgk_ctx* c, void* d_ptr) {
  if (!c || !d_ptr) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  CU(cudaIpcCloseMemHandle(d_ptr));
  return APGK_OK;
}

int apgk_count_pieces_peer(apgk_ctx* c, const void* const* d_src_base, uint32_t n_src, const uint32_t* d_sizes_all,
                           const uint64_t* src_off, uint64_t bucket_lo, uint64_t bucket_hi, int32_t split_bits,
                           const uint32_t* d_sub_sizes) {
  if (!c || !d_src_base || !d_sizes_all || !src_off || n_src == 0 || n_src > 1024) return APGK_E_ARG;
  c->gen++;
  CU(cudaSetDevice(c->device));
  std::vector<const void*> bases(d_src_base, d_src_base + n_src);
  for (uint32_t s = 0; s < n_src; s++)
    if (!bases[s]) bases[s] = c->B.p;  // NULL = this rank's own partition buffer
  switch (c->W) {
    case 1: return count_pieces_impl<1>(c, bases.data(), true, n_src, d_sizes_all, src_off, bucket_lo, bucket_hi, split_bits, d_sub_sizes);
    case 2: return count_pieces_impl<2>(c, bases.data(), true, n_src, d_sizes_all, src_off, bucket_lo, bucket_hi, split_bits, d_sub_sizes);
    case 3: return count_pieces_impl<3>(c, bases.data(), true, n_src, d_sizes_all, src_off, bucket_lo, bucket_hi, split_bits, d_sub_sizes);
  }
  return APGK_E_ARG;
}

int apgk_totals(const apgk_ctx* c, uint64_t* n_instances, uint64_t* n_distinct) {
  if (!c) return APGK_E_ARG;
  if (!c->finished) return APGK_E_STATE;
  if (n_instances) *n_instances = c->n_instances;
  if (n_distinct) *n_distinct = c->n_distinct;
  return APGK_OK;
}

int apgk_spectrum_sparse(apgk_ctx* c, const uint64_t** freq, const uint64_t** n_kmers, uint64_t* n) {
  if (!c) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  int rc = load_spectrum(c);
  if (rc) return rc;
  if (freq) *freq = c->sparse_f.data();
  if (n_kmers) *n_kmers = c->sparse_n.data();
  if (n) *n = c->sparse_f.size();
  return APGK_OK;
}

int apgk_spectrum(apgk_ctx* c, const uint64_t** spec, uint64_t* len) {
  if (!c || !spec || !len) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  int rc = load_spectrum(c);
  if (rc) return rc;
  if (c->spec_host.empty()) {
    const uint64_t mx = c->sparse_f.empty() ? 0 : c->sparse_f.back();
    if (mx + 1 > (1ull << 28)) FAIL(APGK_E_RANGE, "largest count %llu: use apgk_spectrum_sparse", (unsigned long long)mx);
    c->spec_host.assign(mx + 1, 0);
    for (size_t i = 0; i < c->sparse_f.size(); i++) c->spec_host[c->sparse_f[i]] = c->sparse_n[i];
  }
  *spec = c->spec_host.data();
  *len = c->spec_host.size();
  return APGK_OK;
}

int apgk_counts_device(apgk_ctx* c, const uint64_t** d_kmers, const uint32_t** d_counts, uint64_t* n_distinct) {
  if (!c) return APGK_E_ARG;
  if (!c->finished || !c->have_table) FAIL(APGK_E_STATE, "no table: finish with APGK_WANT_COUNTS first");
  if (d_kmers) *d_kmers = c->out_keys.as<uint64_t>();
  if (d_counts) *d_counts = c->out_cnt.as<uint32_t>();
  if (n_distinct) *n_distinct = c->n_distinct;
  return APGK_OK;
}

int apgk_counts_copy(apgk_ctx* c, uint64_t first, uint64_t n, uint64_t* kmers_out, uint32_t* counts_out) {
  if (!c) return APGK_E_ARG;
  if (!c->finished || !c->have_table) FAIL(APGK_E_STATE, "no table: finish with APGK_WANT_COUNTS first");
  if (first + n > c->n_distinct) FAIL(APGK_E_ARG, "range beyond the table");
  if (!n) return APGK_OK;
  CU(cudaSetDevice(c->device));
  const size_t kb = (size_t)c->W * 8;
  if (kmers_out) CU(cudaMemcpyAsync(kmers_out, c->out_keys.as<unsigned char>() + first * kb, n * kb, cudaMemcpyDeviceToHost, c->stream));
  if (counts_out) CU(cudaMemcpyAsync(counts_out, c->out_cnt.as<uint32_t>() + first, n * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return APGK_OK;
}

int apgk_release_temp(apgk_ctx* c) {
  if (!c) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  { int rc = wait_ingest(c); if (rc) return rc; }
  CU(cudaStreamSynchronize(c->stream));
  // B and sub_sizes stay: the peers of a group may have them mapped
  DevBuf* tmp[] = {&c->A, &c->T, &c->C2, &c->TK, &c->scratch, &c->stacks, &c->chunksum, &c->chunksum0, &c->piece_off, &c->piece_tmp,
                   &c->occ, &c->occ_pos, &c->occ_tmp, &c->staging};
  for (DevBuf* b : tmp) b->release();
  c->hp0_elems = ~0ull;            // the level-0 plan's chunk rows went with chunksum0
  c->have_occ = false; c->n_occ = 0;
  c->part_ready = false; c->part_n = 0;
  c->tmp_keys_last = nullptr;
  return APGK_OK;
}

int apgk_reserve_table(apgk_ctx* c, uint64_t n_records) {
  if (!c) return APGK_E_ARG;
  c->gen++;
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  const size_t kb = (size_t)c->W * 8;
  if (c->out_keys.cap < n_records * kb || c->out_cnt.cap < n_records * 4) {
    // the table's present contents are not kept: this is a sizing hint given before a count
    c->out_keys.release(); c->out_cnt.release();
    CU(c->out_keys.ensure(std::max<size_t>(n_records, 1) * kb));
    CU(c->out_cnt.ensure(std::max<size_t>(n_records, 1) * 4));
    c->have_table = false;
  }
  return APGK_OK;
}

int apgk_prefix_range(apgk_ctx* c, int32_t prefix_bits, uint64_t prefix, uint64_t* first, uint64_t* n) {
  if (!c || !first || !n) return APGK_E_ARG;
  if (!c->finished || !c->have_table) FAIL(APGK_E_STATE, "no table: finish with APGK_WANT_COUNTS first");
  const int P = c->geom.D0 + c->geom.D1;
  if (prefix_bits < 0 || prefix_bits > P || c->geom.pad != 0 || (prefix >> prefix_bits) != 0)
    FAIL(APGK_E_ARG, "apgk_prefix_range: prefix_bits must be 0..%d (the table's index bits) and the prefix below 2^prefix_bits", P);
  *first = 0; *n = 0;
  if (!c->n_distinct) return APGK_OK;
  CU(cudaSetDevice(c->device));
  unsigned long long lo = 0, hi = 0;
  const unsigned long long* idx = c->out_off.as<unsigned long long>();
  CU(cudaMemcpyAsync(&lo, idx + (prefix << (P - prefix_bits)), 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(&hi, idx + ((prefix + 1) << (P - prefix_bits)), 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  *first = lo; *n = hi - lo;
  return APGK_OK;
}

int apgk_lookup(apgk_ctx* c, const uint64_t* kmers, uint64_t n, int canonicalise, uint32_t* counts_out) {
  if (!c || (!kmers && n) || (!counts_out && n)) return APGK_E_ARG;
  if (!c->finished || !c->have_table) FAIL(APGK_E_STATE, "no table: finish with APGK_WANT_COUNTS first");
  CU(cudaSetDevice(c->device));
  switch (c->W) {
    case 1: return lookup_impl<1>(c, kmers, n, canonicalise, counts_out);
    case 2: return lookup_impl<2>(c, kmers, n, canonicalise, counts_out);
    case 3: return lookup_impl<3>(c, kmers, n, canonicalise, counts_out);
  }
  return APGK_E_ARG;
}

int apgk_read_freqs(apgk_ctx* c, uint64_t first_base, uint64_t n_bases, uint32_t* out) {
  if (!c || (!out && n_bases)) return APGK_E_ARG;
  if (!c->finished || !c->have_table) FAIL(APGK_E_STATE, "no table: finish with APGK_WANT_COUNTS first");
  if (first_base + n_bases > c->total_bases) FAIL(APGK_E_ARG, "range beyond the read store");
  CU(cudaSetDevice(c->device));
  if (first_base == 0 && n_bases == c->total_bases && n_bases && c->table_from_reads && !kFreqDirect) {
    // the whole store: bulk form (bucket scatter + per-bucket placement) into a device buffer, then one copy
    CU(c->occ_tmp.ensure(n_bases * 4));
    int rc = read_freqs_bulk_dispatch(c, c->occ_tmp.as<uint32_t>());
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, c->occ_tmp.p, n_bases * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return APGK_OK;
  }
  switch (c->W) {
    case 1: return read_freqs_impl<1>(c, first_base, n_bases, out);
    case 2: return read_freqs_impl<2>(c, first_base, n_bases, out);
    case 3: return read_freqs_impl<3>(c, first_base, n_bases, out);
  }
  return APGK_E_ARG;
}

int apgk_build_occurrences(apgk_ctx* c) {
  if (!c) return APGK_E_ARG;
  if (!c->finished || !c->have_table) FAIL(APGK_E_STATE, "no table: finish with APGK_WANT_COUNTS first");
  if (!c->table_from_reads)
    FAIL(APGK_E_STATE, "occurrences need a table counted from this context's read store (apgk_finish, not a shard or a key array)");
  if (c->n_reads > 0xFFFFFFFFull) FAIL(APGK_E_RANGE, "occurrences: read ids are 32-bit, %llu reads", (unsigned long long)c->n_reads);
  CU(cudaSetDevice(c->device));
  switch (c->W) {
    case 1: return c->geom.REM <= 32 ? build_occurrences_impl<1, uint32_t>(c) : build_occurrences_impl<1, Key<1>>(c);
    case 2: return build_occurrences_impl<2, Key<2>>(c);
    case 3: return build_occurrences_impl<3, Key<3>>(c);
  }
  return APGK_E_ARG;
}

int apgk_occurrences_info(const apgk_ctx* c, uint64_t* n_occ, uint64_t* n_big_runs, float* ms5) {
  if (!c) return APGK_E_ARG;
  if (!c->have_occ) return APGK_E_STATE;
  if (n_occ) *n_occ = c->n_occ;
  if (n_big_runs) *n_big_runs = c->n_big_runs;
  if (ms5) for (int i = 0; i < 5; i++) ms5[i] = c->occ_ms[i];
  return APGK_OK;
}

int apgk_occurrences_device(apgk_ctx* c, const uint64_t** d_run_off, const uint64_t** d_occ, uint64_t* n_occ) {
  if (!c) return APGK_E_ARG;
  if (!c->have_occ) FAIL(APGK_E_STATE, "no occurrences: call apgk_build_occurrences first");
  if (d_run_off) *d_run_off = c->occ_off.as<uint64_t>();
  if (d_occ) *d_occ = c->n_occ ? c->occ.as<uint64_t>() : nullptr;
  if (n_occ) *n_occ = c->n_occ;
  return APGK_OK;
}

int apgk_occurrences_copy(apgk_ctx* c, uint64_t first_kmer, uint64_t n_kmers, uint64_t* run_off_out, uint32_t* read_id_out,
                          int32_t* pos_out) {
  if (!c) return APGK_E_ARG;
  if (!c->have_occ) FAIL(APGK_E_STATE, "no occurrences: call apgk_build_occurrences first");
  if (first_kmer > c->n_distinct || n_kmers > c->n_distinct - first_kmer) FAIL(APGK_E_ARG, "k-mer range beyond the table");
  CU(cudaSetDevice(c->device));
  return occurrences_copy_impl(c, first_kmer, n_kmers, run_off_out, read_id_out, pos_out);
}

int apgk_read_freqs_device(apgk_ctx* c, uint32_t* d_out, float* ms3) {
  if (!c || !d_out) return APGK_E_ARG;
  if (!c->finished || !c->have_table) FAIL(APGK_E_STATE, "no table: finish with APGK_WANT_COUNTS first");
  if (!c->table_from_reads)
    FAIL(APGK_E_STATE, "the bulk form needs a table counted from this context's read store (apgk_finish, not a shard or a key array)");
  CU(cudaSetDevice(c->device));
  for (float& m : c->freq_ms) m = 0;
  int rc;
  if (kFreqDirect) {   // the per-window table search, for comparison
    { int r2 = wait_ingest(c); if (r2) return r2; }
    for (cudaEvent_t& e : c->occ_ev) if (!e) CU(cudaEventCreate(&e));
    CU(cudaEventRecord(c->occ_ev[0], c->stream));
    constexpr int NT = 128;
    const uint64_t threads = (c->total_bases + POS_PER_THREAD - 1) / POS_PER_THREAD;
    if (threads) {
      switch (c->W) {
        case 1: k_read_freqs<1, NT><<<(unsigned)((threads + NT - 1) / NT), NT, 0, c->stream>>>(read_store(c), freq_table<1>(c), 0, c->total_bases, d_out); break;
        case 2: k_read_freqs<2, NT><<<(unsigned)((threads + NT - 1) / NT), NT, 0, c->stream>>>(read_store(c), freq_table<2>(c), 0, c->total_bases, d_out); break;
        case 3: k_read_freqs<3, NT><<<(unsigned)((threads + NT - 1) / NT), NT, 0, c->stream>>>(read_store(c), freq_table<3>(c), 0, c->total_bases, d_out); break;
      }
      LAUNCHED();
    }
    CU(cudaEventRecord(c->occ_ev[1], c->stream));
    CU(cudaStreamSynchronize(c->stream));
    cudaEventElapsedTime(&c->freq_ms[1], c->occ_ev[0], c->occ_ev[1]);
    rc = APGK_OK;
  } else {
    rc = read_freqs_bulk_dispatch(c, d_out);
  }
  if (ms3) for (int i = 0; i < 3; i++) ms3[i] = c->freq_ms[i];
  return rc;
}

int apgk_owner_plan(apgk_ctx* c, uint32_t n_ranks, uint64_t* counts_out) {
  if (!c || !counts_out || n_ranks < 1 || n_ranks > 1024) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  switch (c->W) {
    case 1: return owner_plan_impl<1>(c, n_ranks, counts_out);
    case 2: return owner_plan_impl<2>(c, n_ranks, counts_out);
    case 3: return owner_plan_impl<3>(c, n_ranks, counts_out);
  }
  return APGK_E_ARG;
}

int apgk_owner_scatter(apgk_ctx* c, uint64_t* d_keys_out) {
  if (!c) return APGK_E_ARG;
  if (!c->owner_ranks) FAIL(APGK_E_STATE, "apgk_owner_plan has not run");
  CU(cudaSetDevice(c->device));
  switch (c->W) {
    case 1: return owner_scatter_impl<1>(c, d_keys_out);
    case 2: return owner_scatter_impl<2>(c, d_keys_out);
    case 3: return owner_scatter_impl<3>(c, d_keys_out);
  }
  return APGK_E_ARG;
}

int apgk_key_buffer(apgk_ctx* c, uint64_t n_keys, uint64_t** d_ptr) {
  if (!c || !d_ptr) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  CU(c->A.ensure(std::max<size_t>(n_keys, 1) * (size_t)c->W * 8));
  *d_ptr = c->A.as<uint64_t>();
  return APGK_OK;
}

int apgk_owner_of(int K, const uint64_t* kmers, uint64_t n, uint32_t n_ranks, uint32_t* owner_out) {
  if (K < 1 || K > APGK_MAX_K || !kmers || !owner_out || !n_ranks) return APGK_E_ARG;
  const int W = words_for(K);
  for (uint64_t i = 0; i < n; i++) {
    if (W == 1) { Key<1> k; k.w[0] = kmers[i]; owner_out[i] = key_owner(k, n_ranks); }
    else if (W == 2) { Key<2> k; k.w[0] = kmers[2 * i]; k.w[1] = kmers[2 * i + 1]; owner_out[i] = key_owner(k, n_ranks); }
    else { Key<3> k; k.w[0] = kmers[3 * i]; k.w[1] = kmers[3 * i + 1]; k.w[2] = kmers[3 * i + 2]; owner_out[i] = key_owner(k, n_ranks); }
  }
  return APGK_OK;
}

int apgk_spectrum_device(apgk_ctx* c, uint64_t** d_spec, uint64_t* len) {
  if (!c || !d_spec) return APGK_E_ARG;
  if (!c->finished) FAIL(APGK_E_STATE, "apgk_finish has not run");
  *d_spec = c->spec_dense.as<uint64_t>();
  if (len) *len = SPEC_DENSE;
  return APGK_OK;
}

int apgk_spectrum_reload(apgk_ctx* c) {
  if (!c) return APGK_E_ARG;
  c->spec_loaded = false;
  c->spec_host.clear();
  return APGK_OK;
}

int apgk_stage_ms(const apgk_ctx* c, float* ms_out) {
  if (!c || !ms_out) return APGK_E_ARG;
  for (int s = 0; s < APGK_N_STAGES; s++) ms_out[s] = c->stage_ms[s];
  return APGK_OK;
}
const char* apgk_stage_name(int i) { return (i >= 0 && i < APGK_N_STAGES) ? kStageNames[i] : ""; }
uint64_t apgk_kernel_launches(const apgk_ctx* c) { return c ? c->launches : 0; }
void apgk_reset_counters(apgk_ctx* c) { if (c) c->launches = 0; }

int apgk_geometry(const apgk_ctx* c, int32_t* out8) {
  if (!c || !out8) return APGK_E_ARG;
  out8[0] = c->geom.D0; out8[1] = c->geom.D1; out8[2] = c->geom.REM; out8[3] = (int32_t)c->elem_bytes;
  out8[4] = (int32_t)std::min<uint64_t>(c->n_big, 0x7fffffff);
  out8[5] = (int32_t)std::min<uint32_t>(c->n_deferred, 0x7fffffff);
  out8[6] = (int32_t)c->local_max;
  out8[7] = (int32_t)c->n_rounds;
  return APGK_OK;
}

int apgk_device_alloc(apgk_ctx* c, void** p, size_t bytes) {
  if (!c || !p) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  CU(cudaMalloc(p, bytes ? bytes : 1));
  return APGK_OK;
}
int apgk_device_free(apgk_ctx* c, void* p) {
  if (!c) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  CU(cudaFree(p));
  return APGK_OK;
}
int apgk_device_copy_to_host(apgk_ctx* c, void* dst_host, const void* src_dev, size_t bytes) {
  if (!c || (!dst_host && bytes)) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  if (bytes) {
    CU(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  return APGK_OK;
}

int apgk_host_alloc(void** p, size_t bytes) {
  if (!p) return APGK_E_ARG;
  return cudaHostAlloc(p, bytes, cudaHostAllocDefault) == cudaSuccess ? APGK_OK : APGK_E_NOMEM;
}
int apgk_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? APGK_OK : APGK_E_CUDA; }


// ---------------------------------------------------------------- groups
int apgk_group_unique_id(uint8_t id_out[APGK_GROUP_ID_BYTES]) {
  if (!id_out) return APGK_E_ARG;
  static_assert(sizeof(ncclUniqueId) == APGK_GROUP_ID_BYTES, "unique id size");
  if (!g_nccl.load().empty()) return APGK_E_CUDA;
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return APGK_E_CUDA;
  memcpy(id_out, &id, APGK_GROUP_ID_BYTES);
  return APGK_OK;
}

static int group_init_rank(apgk_group* g, RankState& r, apgk_ctx* c) {
  if (c->group) GFAIL(APGK_E_STATE, "the context already belongs to a group");
  r.c = c;
  c->group = g;
  GCU(cudaSetDevice(c->device));
  GCU(cudaEventCreateWithFlags(&r.ev_a, cudaEventDisableTiming));
  GCU(cudaEventCreateWithFlags(&r.ev_b, cudaEventDisableTiming));
  return APGK_OK;
}

int apgk_group_join(apgk_ctx* ctx, const uint8_t id[APGK_GROUP_ID_BYTES], int32_t rank, int32_t world, apgk_group** out) {
  if (!ctx || !id || !out || world < 1 || world > 1024 || rank < 0 || rank >= world) return APGK_E_ARG;
  *out = nullptr;
  apgk_ctx* c = ctx;
  const std::string e = g_nccl.load();
  if (!e.empty()) FAIL(APGK_E_CUDA, "%s", e.c_str());
  apgk_group* g = new apgk_group();
  g->world = world; g->n_local = 1; g->rank0 = rank; g->use_nccl = true;
  g->rs.resize(1);
  int rc = group_init_rank(g, g->rs[0], ctx);
  if (rc == APGK_OK) {
    ncclUniqueId nid;
    memcpy(&nid, id, APGK_GROUP_ID_BYTES);
    const ncclResult_t r = g_nccl.CommInitRank(&g->comm, world, nid, rank);
    if (r != ncclSuccess) { g->err = std::string("ncclCommInitRank failed: ") + g_nccl.GetErrorString(r); rc = APGK_E_CUDA; }
  }
  if (rc) { c->err = g->err; apgk_group_destroy(g); return rc; }
  *out = g;
  return APGK_OK;
}

int apgk_group_local(apgk_ctx* const* ctxs, int32_t n, apgk_group** out) {
  if (!ctxs || !out || n < 1 || n > 1024) return APGK_E_ARG;
  *out = nullptr;
  for (int i = 0; i < n; i++) if (!ctxs[i]) return APGK_E_ARG;
  apgk_group* g = new apgk_group();
  g->world = n; g->n_local = n; g->rank0 = 0; g->use_nccl = false;
  g->rs.resize(n);
  int rc = APGK_OK;
  for (int i = 0; i < n && rc == APGK_OK; i++) rc = group_init_rank(g, g->rs[i], ctxs[i]);
  // contexts on different devices read each other's partition buffers directly
  for (int i = 0; i < n && rc == APGK_OK; i++)
    for (int j = 0; j < n; j++) {
      const int di = ctxs[i]->device, dj = ctxs[j]->device;
      if (di == dj) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, di, dj);
      if (!can) { g->err = "devices of a single-process group must be peer-accessible"; rc = APGK_E_CUDA; break; }
      cudaSetDevice(di);
      const cudaError_t e = cudaDeviceEnablePeerAccess(dj, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { g->err = cudaGetErrorString(e); rc = APGK_E_CUDA; break; }
      cudaGetLastError();
    }
  if (rc) { ctxs[0]->err = g->err; apgk_group_destroy(g); return rc; }
  *out = g;
  return APGK_OK;
}

void apgk_group_destroy(apgk_group* g) {
  if (!g) return;
  for (size_t i = 0; i < g->rs.size(); i++)
    if (g->rs[i].c) group_detach(g, g->rs[i].c);
  if (g->comm) g_nccl.CommDestroy(g->comm);
  delete g;
}

const char* apgk_group_last_error(const apgk_group* g) { return g ? g->err.c_str() : "null group"; }

int apgk_group_count(apgk_group* g) {
  if (!g) return APGK_E_ARG;
  return group_count(g);
}

int apgk_group_read_freqs_device(apgk_group* g, uint32_t* const* d_out, const uint64_t* first_base, const uint64_t* n_bases,
                                 apgk_group_freq_stats* stats) {
  if (!g) return APGK_E_ARG;
  return group_read_freqs(g, d_out, first_base, n_bases, stats);
}

int apgk_group_totals(const apgk_group* g, uint64_t* n_instances, uint64_t* n_distinct) {
  if (!g) return APGK_E_ARG;
  if (!g->counted) return APGK_E_STATE;
  if (n_instances) *n_instances = g->n_instances;
  if (n_distinct) *n_distinct = g->n_distinct;
  return APGK_OK;
}

int apgk_group_spectrum_sparse(apgk_group* g, const uint64_t** freq, const uint64_t** n_kmers, uint64_t* n) {
  if (!g) return APGK_E_ARG;
  if (!g->counted) GFAIL(APGK_E_STATE, "apgk_group_count has not run");
  if (freq) *freq = g->sparse_f.data();
  if (n_kmers) *n_kmers = g->sparse_n.data();
  if (n) *n = g->sparse_f.size();
  return APGK_OK;
}

int apgk_group_stats_get(const apgk_group* g, apgk_group_stats* out) {
  if (!g || !out) return APGK_E_ARG;
  if (!g->counted) return APGK_E_STATE;
  *out = g->stats;
  return APGK_OK;
}

// ---------------------------------------------------------------- host test hooks
int apgk_debug_counters(apgk_ctx* c, uint64_t* out8, int reset) {
  if (!c || !out8) return APGK_E_ARG;
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaMemcpyFromSymbol(out8, g_l4_dbg, 64));
  if (reset) { unsigned long long z[8] = {0}; CU(cudaMemcpyToSymbol(g_l4_dbg, z, 64)); }
  return APGK_OK;
}

int apgk_debug_host_extract(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, int K, uint64_t* kmers_out,
                            uint8_t* valid_out) {
  if (!packed || !off || K < 1 || K > APGK_MAX_K) return APGK_E_ARG;
  if (!n_reads) return APGK_OK;
  switch (words_for(K)) {
    case 1: host_extract<1>(packed, off, n_reads, K, kmers_out, valid_out); break;
    case 2: host_extract<2>(packed, off, n_reads, K, kmers_out, valid_out); break;
    case 3: host_extract<3>(packed, off, n_reads, K, kmers_out, valid_out); break;
  }
  return APGK_OK;
}

int apgk_debug_host_topdigits(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, int K, int D,
                              uint32_t* digits_out) {
  if (!packed || !off || !digits_out || K < 1 || K > APGK_MAX_K || D < 1 || D > 16 || K < (D + 1) / 2 || 2 * K < D)
    return APGK_E_ARG;
  if (!n_reads) return APGK_OK;
  const uint64_t b0 = off[0], total = off[n_reads] - b0;
  std::vector<uint32_t> bases((total + 15) / 16 + 16, 0);
  for (uint64_t q = 0; q < total; q++) {
    const uint64_t s = b0 + q;
    bases[q >> 4] |= (uint32_t)((packed[s >> 2] >> ((s & 3) * 2)) & 3u) << ((q & 15) * 2);
  }
  for (uint64_t p = 0; p < total; p += 16)
    top_digits16(bases.data(), p, K, D, [&](int j, uint32_t d) { if (p + j < total) digits_out[p + j] = d; });
  return APGK_OK;
}

int apgk_debug_host_canonical(int K, const uint64_t* kmers, uint64_t n, uint64_t* out) {
  if (K < 1 || K > APGK_MAX_K) return APGK_E_ARG;
  const int W = words_for(K);
  for (uint64_t i = 0; i < n; i++) {
    if (W == 1) { Key<1> k; k.w[0] = kmers[i]; k = key_canonical(k, K); out[i] = k.w[0]; }
    else if (W == 2) { Key<2> k; memcpy(k.w, kmers + 2 * i, 16); k = key_canonical(k, K); memcpy(out + 2 * i, k.w, 16); }
    else { Key<3> k; memcpy(k.w, kmers + 3 * i, 24); k = key_canonical(k, K); memcpy(out + 3 * i, k.w, 24); }
  }
  return APGK_OK;
}

int apgk_debug_host_table_find(int K, const uint64_t* sorted_kmers, uint64_t n, int prefix_bits, const uint64_t* queries,
                               uint64_t n_q, uint64_t* idx_out) {
  if (K < 1 || K > APGK_MAX_K || prefix_bits < 1 || prefix_bits > 24) return APGK_E_ARG;
  if (words_for(K) > 1 && prefix_bits > 2 * K) return APGK_E_ARG;
  switch (words_for(K)) {
    case 1: host_table_find<1>(K, sorted_kmers, n, prefix_bits, queries, n_q, idx_out); break;
    case 2: host_table_find<2>(K, sorted_kmers, n, prefix_bits, queries, n_q, idx_out); break;
    case 3: host_table_find<3>(K, sorted_kmers, n, prefix_bits, queries, n_q, idx_out); break;
  }
  return APGK_OK;
}

int apgk_debug_host_splitters(const uint32_t* bucket_sizes, uint32_t n_buckets, uint32_t world, uint32_t bucket_cost, uint32_t* bounds_out) {
  if (!bucket_sizes || !bounds_out || !world) return APGK_E_ARG;
  // what k_total_sizes (cost column) + the scan + k_splitters do on the device, here on the host
  std::vector<unsigned long long> S((size_t)n_buckets + 1, 0);
  for (uint32_t b = 0; b < n_buckets; b++) S[b + 1] = S[b] + (bucket_sizes[b] ? (unsigned long long)bucket_sizes[b] + bucket_cost : 0ull);
  for (uint32_t r = 0; r <= world; r++) bounds_out[r] = splitter_bound(S.data(), n_buckets, world, r);
  return APGK_OK;
}

int apgk_debug_host_synth(const apgk_synth_params* p, uint64_t r0, uint64_t n_reads, uint8_t* packed_out) {
  if (!p || !packed_out) return APGK_E_ARG;
  SynthParams sp{p->genome_len, p->seed_g, p->seed_p, p->seed_q, p->seed_r, p->seed_e, p->read_len, p->err_per_200};
  const uint64_t nb = n_reads * (uint64_t)p->read_len;
  uint32_t* w = (uint32_t*)packed_out;
  for (uint64_t wi = 0; wi * 16 < nb; wi++) w[wi] = synth_word(sp, r0, wi * 16, nb);
  return APGK_OK;
}

}  // extern "C"
