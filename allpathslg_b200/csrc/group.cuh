// group.cuh -- sharded counting behind the C ABI (include/apgk.h "a GROUP of ranks"); part of apgk.cu's
// translation unit.
//
// SURVEY.md section 8(e): the path shards by canonical k-mer with ONE exchange.  apgk_group_count drives, for
// every rank of the group,
//
//   levels 0 + 1 over the rank's reads            (level0_hist / level0_scatter / level1: the single-GPU kernels;
//                                                  the level-1 histogram also leaves the sub-bucket sizes)
//   all-gather of the 2^P bucket sizes            (NCCL, or peer copies inside one process)
//   balanced contiguous bucket ranges             (k_total_sizes -> scan -> k_splitters, on the device)
//   ONE host round trip                           (bounds + shard size: the buffers of the shard are sized)
//   the exchange, fused into the gather kernel    (k_gather_split reads the peers' partition buffers and their
//                                                  sub-bucket counts straight over NVLink peer memory)
//   per-bucket counting of the owned range        (count_buckets: k_local3 & co, table appended)
//   spectrum + totals all-reduce                  (also the barrier that frees the partition buffers)
//
// in k-mer-space rounds when the k-mers of a rank do not fit its device at once: OUTER rounds extract a range of
// level-0 buckets once, INNER rounds run level 1 + exchange + counting over sub-ranges of the extracted keys.
// All ranks cut the rounds from the same all-reduced numbers, so they walk the same ranges.
//
// The driver is a phase machine over the group's LOCAL contexts: one per process in the multi-process form
// (collectives = NCCL, peers' buffers = CUDA IPC mappings), all of them in the single-process form (collectives =
// copies and kernels ordered by events; peers' buffers = plain pointers).  The same code path serves both, which
// is also how the N-rank pipeline is tested on one GPU.
#pragma once
#include <dlfcn.h>
#include <nccl.h>   // types and enums only: the functions are resolved at run time (no link-time dependency)

namespace {

struct NcclApi {
  void* h = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string load() {   // "" or what went wrong
    if (h) return "";
    // a process that already carries an NCCL (PyTorch's bundled one, say) gets that copy: same SONAME
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
      h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (h) break;
    }
    if (!h) return std::string("cannot load libnccl.so.2: ") + dlerror();
    auto sym = [&](const char* n) { return dlsym(h, n); };
    GetUniqueId = (decltype(GetUniqueId))sym("ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))sym("ncclCommInitRank");
    CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
    AllGather = (decltype(AllGather))sym("ncclAllGather");
    AllReduce = (decltype(AllReduce))sym("ncclAllReduce");
    GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
    if (!GetUniqueId || !CommInitRank || !CommDestroy || !AllGather || !AllReduce || !GetErrorString) {
      h = nullptr;
      return "libnccl.so.2 lacks a required symbol";
    }
    return "";
  }
};
NcclApi g_nccl;

constexpr uint32_t OVF_SHIP = 1022;   // spectrum overflow entries (counts >= 65536) a rank ships with the first gather

struct GroupMeta {   // what every rank tells the others before a step (all-gathered, host side)
  uint64_t n_windows, budget, cap_B, cap_sub, ptr_B, ptr_sub, max_round_keys, max_inner_keys;
  int32_t K, flags, prefix_bits, pad_;
};

struct RankState {   // per LOCAL context
  apgk_ctx* c = nullptr;
  DevBuf sizes32, sizes_all, tot32, E_tot, cost32, E_cost, plan_dev, ptrs_dev, red_in, red_out, ovf_out, ovf_all, tot0_red, meta_dev, meta_all, bar;
  unsigned long long* host = nullptr;          // pinned: plan block | reduced spectrum | overflow lists (see offsets)
  size_t host_words = 0;
  std::vector<void*> peer_B, peer_sub;          // [world] device pointers valid on this rank's device (own slot: own buffer)
  std::vector<std::array<uint8_t, 64>> map_hB, map_hS;   // multi-process form: the handle each mapping came from
  std::vector<bool> mapped;
  std::vector<uint64_t> map_pB, map_pS;         // the owner's own pointer values when the mapping was made
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;   // single-process form: cross-rank ordering
  KeyGeom geom_part{}, geom_shard{};
  uint32_t nb = 0, nbf = 0;
  uint64_t n_prev = 0, shard_n = 0, remote_bytes = 0;
  std::vector<uint64_t> tot0;                   // own level-0 totals (multi-round steps)
  uint64_t gen_counted = 0;                     // the context's generation when the last count finished
  DevBuf gpos, gcnt;                            // lookups: batch-relative position per slot of B; counters
  cudaEvent_t gev[6]{};                         // lookups: stage boundaries of a batch, start and end of the call
};

}  // namespace

struct apgk_group {
  int world = 1, n_local = 1, rank0 = 0;
  bool use_nccl = false;
  ncclComm_t comm = nullptr;
  std::vector<RankState> rs;
  std::string err;
  // global results of the last count
  std::vector<uint64_t> sparse_f, sparse_n;
  uint64_t n_instances = 0, n_distinct = 0;
  apgk_group_stats stats{};
  bool counted = false;
  // who owns what after the last count: (bucket_lo, bucket_hi, owner) over the 2^P coarse buckets of every inner
  // round; they tile [0, 2^P).  freq_ready: that count kept tables (APGK_WANT_COUNTS), lookups can be made.
  std::vector<std::array<uint32_t, 3>> own_segs;
  bool freq_ready = false;
  bool dead = false;   // a member context was destroyed: the group can only be destroyed
};

namespace {

#define GFAIL(code, ...)                       \
  do {                                         \
    char b__[512];                             \
    snprintf(b__, sizeof b__, __VA_ARGS__);    \
    g->err = b__;                              \
    return (code);                             \
  } while (0)
#define GCU(call)                                                                                        \
  do {                                                                                                   \
    cudaError_t e__ = (call);                                                                            \
    if (e__ != cudaSuccess) {                                                                            \
      char b__[512];                                                                                     \
      snprintf(b__, sizeof b__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
      g->err = b__;                                                                                      \
      return (e__ == cudaErrorMemoryAllocation) ? APGK_E_NOMEM : APGK_E_CUDA;                            \
    }                                                                                                    \
  } while (0)
#define GNCCL(call)                                                                                      \
  do {                                                                                                   \
    ncclResult_t r__ = (call);                                                                           \
    if (r__ != ncclSuccess) {                                                                            \
      char b__[512];                                                                                     \
      snprintf(b__, sizeof b__, "%s failed: %s (%s:%d)", #call, g_nccl.GetErrorString(r__), __FILE__, __LINE__); \
      g->err = b__;                                                                                      \
      return APGK_E_CUDA;                                                                                \
    }                                                                                                    \
  } while (0)
// a context-level call inside the group: its message becomes the group's
#define GCTX(c, call)                                  \
  do {                                                 \
    int rc__ = (call);                                 \
    if (rc__) { g->err = (c)->err; return rc__; }      \
  } while (0)

// ---------------------------------------------------------------- collectives over the group's local contexts
// Every helper is called once per phase with per-local-rank arguments.

// bytes from every rank, host side (blocking).  mine: n_local blocks of `bytes`; all: world blocks.
int coll_allgather_host(apgk_group* g, const void* mine, size_t bytes, void* all) {
  if (!g->use_nccl) { memcpy(all, mine, bytes * g->n_local); return APGK_OK; }
  RankState& r = g->rs[0];
  apgk_ctx* c = r.c;
  GCU(cudaSetDevice(c->device));
  GCU(r.meta_dev.ensure(bytes));
  GCU(r.meta_all.ensure(bytes * g->world));
  GCU(cudaMemcpyAsync(r.meta_dev.p, mine, bytes, cudaMemcpyHostToDevice, c->stream));
  GNCCL(g_nccl.AllGather(r.meta_dev.p, r.meta_all.p, bytes, ncclUint8, g->comm, c->stream));
  GCU(cudaMemcpyAsync(all, r.meta_all.p, bytes * g->world, cudaMemcpyDeviceToHost, c->stream));
  GCU(cudaStreamSynchronize(c->stream));
  return APGK_OK;
}

// single-process form: every local stream waits until all local streams have reached this point
int local_cross_wait(apgk_group* g, bool use_b) {
  for (RankState& r : g->rs) {
    GCU(cudaSetDevice(r.c->device));
    GCU(cudaEventRecord(use_b ? r.ev_b : r.ev_a, r.c->stream));
  }
  for (RankState& r : g->rs) {
    GCU(cudaSetDevice(r.c->device));
    for (RankState& s : g->rs)
      if (&s != &r) GCU(cudaStreamWaitEvent(r.c->stream, use_b ? s.ev_b : s.ev_a, 0));
  }
  return APGK_OK;
}

// device all-gather: src(i) = `bytes` on local rank i  ->  dst(i) = world * bytes on every local rank, stream ordered
template <typename FS, typename FD>
int coll_allgather_dev(apgk_group* g, size_t bytes, FS src, FD dst) {
  if (g->use_nccl) {
    RankState& r = g->rs[0];
    GCU(cudaSetDevice(r.c->device));
    GNCCL(g_nccl.AllGather(src(0), dst(0), bytes, ncclUint8, g->comm, r.c->stream));
    return APGK_OK;
  }
  { int rc = local_cross_wait(g, false); if (rc) return rc; }
  for (int i = 0; i < g->n_local; i++) {
    GCU(cudaSetDevice(g->rs[i].c->device));
    for (int s = 0; s < g->n_local; s++)
      GCU(cudaMemcpyAsync((unsigned char*)dst(i) + (size_t)s * bytes, src(s), bytes, cudaMemcpyDefault, g->rs[i].c->stream));
  }
  // the sources may not be overwritten before every copy has run
  return local_cross_wait(g, true);
}

// device all-reduce of n u64 (SUM or MAX): in(i) -> out(i) on every local rank, stream ordered
template <typename FI, typename FO>
int coll_allreduce_u64(apgk_group* g, uint64_t n, bool is_max, FI in, FO out) {
  if (g->use_nccl) {
    RankState& r = g->rs[0];
    GCU(cudaSetDevice(r.c->device));
    GNCCL(g_nccl.AllReduce(in(0), out(0), n, ncclUint64, is_max ? ncclMax : ncclSum, g->comm, r.c->stream));
    return APGK_OK;
  }
  { int rc = local_cross_wait(g, false); if (rc) return rc; }
  std::vector<const void*> ptrs(g->n_local);
  for (int s = 0; s < g->n_local; s++) ptrs[s] = in(s);
  for (int i = 0; i < g->n_local; i++) {
    RankState& r = g->rs[i];
    apgk_ctx* c = r.c;
    GCU(cudaSetDevice(c->device));
    GCU(r.ptrs_dev.ensure(3 * (size_t)g->world * 8));
    unsigned char* slot = r.ptrs_dev.as<unsigned char>() + 2 * (size_t)g->world * 8;
    GCU(cudaMemcpyAsync(slot, ptrs.data(), (size_t)g->n_local * 8, cudaMemcpyHostToDevice, c->stream));
    const unsigned grid = (unsigned)((n + 255) / 256);
    if (is_max) k_max_ranks<<<grid, 256, 0, c->stream>>>((const unsigned long long* const*)slot, (uint32_t)g->n_local, n, (unsigned long long*)out(i));
    else k_sum_ranks<<<grid, 256, 0, c->stream>>>((const unsigned long long* const*)slot, (uint32_t)g->n_local, n, (unsigned long long*)out(i));
    c->launches++;
    GCU(cudaGetLastError());
  }
  return local_cross_wait(g, true);
}

// no rank's stream passes this point before every rank's stream has reached it
int coll_barrier_dev(apgk_group* g) {
  if (!g->use_nccl) return local_cross_wait(g, false);
  RankState& r = g->rs[0];
  GCU(cudaSetDevice(r.c->device));
  GCU(r.bar.ensure(16));
  GNCCL(g_nccl.AllReduce(r.bar.p, r.bar.as<unsigned char>() + 8, 1, ncclUint64, ncclSum, g->comm, r.c->stream));
  return APGK_OK;
}

int ceil_log2(int x) { int b = 0; while ((1 << b) < x) b++; return b; }

// ---------------------------------------------------------------- exported buffers of the multi-process form
// B (the partition buffer) and sub_sizes are read by the peers.  They are sized before the exchange of a step
// and never reallocated while a peer has them mapped: every rank knows from the all-gathered capacities which
// ranks must grow theirs, unmaps those, and only after a barrier do the owners reallocate and re-export.
int refresh_exports(apgk_group* g, const std::vector<GroupMeta>& meta, const std::vector<uint64_t>& need_B, uint64_t need_sub) {
  const int world = g->world;
  if (!g->use_nccl) {
    for (RankState& r : g->rs) {
      apgk_ctx* c = r.c;
      GCU(cudaSetDevice(c->device));
      GCU(c->B.ensure(std::max<uint64_t>(need_B[g->rank0 + (&r - &g->rs[0])], 16)));
      GCU(c->sub_sizes.ensure(std::max<uint64_t>(need_sub, 16)));
    }
    for (RankState& r : g->rs) {
      r.peer_B.assign(world, nullptr); r.peer_sub.assign(world, nullptr);
      for (int s = 0; s < world; s++) { r.peer_B[s] = g->rs[s].c->B.p; r.peer_sub[s] = g->rs[s].c->sub_sizes.p; }
    }
    return APGK_OK;
  }
  RankState& r = g->rs[0];
  apgk_ctx* c = r.c;
  const int me = g->rank0;
  GCU(cudaSetDevice(c->device));
  if (r.peer_B.empty()) {
    r.peer_B.assign(world, nullptr); r.peer_sub.assign(world, nullptr);
    r.map_hB.assign(world, {}); r.map_hS.assign(world, {});
    r.mapped.assign(world, false);
    r.map_pB.assign(world, 0); r.map_pS.assign(world, 0);
  }
  bool any = false;
  std::vector<bool> grows(world, false);
  for (int s = 0; s < world; s++) {
    grows[s] = meta[s].cap_B < std::max<uint64_t>(need_B[s], 16) || meta[s].cap_sub < std::max<uint64_t>(need_sub, 16);
    // (a buffer that moved behind the group's back -- the context was also used on its own -- is re-mapped too)
    const bool moved = s != me && r.mapped[s] && (meta[s].ptr_B != r.map_pB[s] || meta[s].ptr_sub != r.map_pS[s]);
    if (moved) grows[s] = true;
    any = any || grows[s] || (s != me && !r.mapped[s]);
  }
  if (!any) { r.peer_B[me] = c->B.p; r.peer_sub[me] = c->sub_sizes.p; return APGK_OK; }
  // 1. unmap the buffers that are about to be reallocated; 2. barrier; 3. owners reallocate; 4. handles travel
  GCU(cudaStreamSynchronize(c->stream));
  for (int s = 0; s < world; s++)
    if (s != me && grows[s] && r.mapped[s]) {
      GCU(cudaIpcCloseMemHandle(r.peer_B[s]));
      GCU(cudaIpcCloseMemHandle(r.peer_sub[s]));
      r.mapped[s] = false;
    }
  { int rc = coll_barrier_dev(g); if (rc) return rc; }
  GCU(cudaStreamSynchronize(c->stream));
  GCU(c->B.ensure(std::max<uint64_t>(need_B[me], 16)));
  GCU(c->sub_sizes.ensure(std::max<uint64_t>(need_sub, 16)));
  struct Handles { uint8_t b[64], s[64]; uint64_t pB, pS; };
  Handles mine{};
  std::vector<Handles> all(world);
  {
    cudaIpcMemHandle_t h;
    GCU(cudaIpcGetMemHandle(&h, c->B.p));
    memcpy(mine.b, &h, 64);
    GCU(cudaIpcGetMemHandle(&h, c->sub_sizes.p));
    memcpy(mine.s, &h, 64);
    mine.pB = (uint64_t)(uintptr_t)c->B.p; mine.pS = (uint64_t)(uintptr_t)c->sub_sizes.p;
  }
  { int rc = coll_allgather_host(g, &mine, sizeof mine, all.data()); if (rc) return rc; }
  for (int s = 0; s < world; s++) {
    if (s == me) { r.peer_B[s] = c->B.p; r.peer_sub[s] = c->sub_sizes.p; continue; }
    const bool same = r.mapped[s] && !memcmp(r.map_hB[s].data(), all[s].b, 64) && !memcmp(r.map_hS[s].data(), all[s].s, 64);
    if (same) continue;
    if (r.mapped[s]) {   // a peer re-exported without announcing it (cannot happen; keep the mapping table honest)
      cudaIpcCloseMemHandle(r.peer_B[s]); cudaIpcCloseMemHandle(r.peer_sub[s]);
      r.mapped[s] = false;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, all[s].b, 64);
    GCU(cudaIpcOpenMemHandle(&r.peer_B[s], h, cudaIpcMemLazyEnablePeerAccess));
    memcpy(&h, all[s].s, 64);
    GCU(cudaIpcOpenMemHandle(&r.peer_sub[s], h, cudaIpcMemLazyEnablePeerAccess));
    memcpy(r.map_hB[s].data(), all[s].b, 64); memcpy(r.map_hS[s].data(), all[s].s, 64);
    r.map_pB[s] = all[s].pB; r.map_pS[s] = all[s].pS;
    r.mapped[s] = true;
  }
  return APGK_OK;
}

// A context leaves its group (apgk_destroy of a context that is still a member, or apgk_group_destroy): its
// mappings of the peers' buffers are closed, the group's per-rank buffers released.  The group stays valid for
// destruction only.
void group_detach(apgk_group* g, apgk_ctx* c) {
  for (RankState& r : g->rs) {
    if (r.c != c) continue;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (g->use_nccl)
      for (size_t s = 0; s < r.mapped.size(); s++)
        if (r.mapped[s]) { cudaIpcCloseMemHandle(r.peer_B[s]); cudaIpcCloseMemHandle(r.peer_sub[s]); r.mapped[s] = false; }
    DevBuf* all[] = {&r.sizes32, &r.sizes_all, &r.tot32, &r.E_tot, &r.cost32, &r.E_cost, &r.plan_dev, &r.ptrs_dev, &r.red_in, &r.red_out, &r.ovf_out,
                     &r.ovf_all, &r.tot0_red, &r.meta_dev, &r.meta_all, &r.bar, &r.gpos, &r.gcnt};
    for (DevBuf* b : all) b->release();
    for (cudaEvent_t& e : r.gev) { if (e) cudaEventDestroy(e); e = nullptr; }
    if (r.host) cudaFreeHost(r.host);
    r.host = nullptr; r.host_words = 0;
    if (r.ev_a) cudaEventDestroy(r.ev_a);
    if (r.ev_b) cudaEventDestroy(r.ev_b);
    r.ev_a = r.ev_b = nullptr;
    r.c = nullptr;
    c->group = nullptr;
    g->dead = true;
  }
}

// layout of RankState::host (pinned), in u64 words
struct HostLayout {
  size_t plan = 0, extra = 0, red = 0, ovf = 0, tot0 = 0, words = 0;
  HostLayout(int world, int bins0) {
    plan = 0;                         // 3 * (world + 1): bounds, E at the bounds, this rank's own prefix at the bounds
    extra = plan + 3 * ((size_t)world + 1);   // 4: flags
    red = extra + 4;                  // SPEC_DENSE + 2: reduced spectrum, n_instances, n_distinct
    ovf = red + SPEC_DENSE + 2;       // world * (1 + OVF_SHIP)
    tot0 = ovf + (size_t)world * (1 + OVF_SHIP);   // 2 * bins0: own totals, max over ranks
    words = tot0 + 2 * (size_t)bins0;
  }
};

struct GRound { int lo, hi; std::vector<std::array<int, 2>> inner; };

// ---------------------------------------------------------------- the step
template <int W, typename ElemB>
int group_count_typed(apgk_group* g, const std::vector<GroupMeta>& meta, bool single, uint64_t cap_outer, uint64_t cap_inner, int d2,
                      uint64_t budget, double inner_bytes) {
  const int world = g->world, nl = g->n_local;
  apgk_ctx* c0 = g->rs[0].c;
  const KeyGeom gp = c0->geom;
  const int bins0 = 1 << gp.D0, bins1 = 1 << gp.D1;
  const uint32_t nb = (uint32_t)bins0 * (uint32_t)bins1, nbf = nb << d2;
  const int want_table = (c0->cfg.flags & APGK_WANT_COUNTS) ? 1 : 0;
  int local_max = std::is_same<ElemB, uint32_t>::value ? LM_U32 : (use_local4(W) ? LM_KEY4 : Geo<W>::LM_KEY);
  if (std::is_same<ElemB, uint32_t>::value) {
    if (const char* e = getenv("APGK_LM")) { if (atoi(e) >= 256 && atoi(e) <= 12288) local_max = atoi(e); }
  }
  // The ranges the ranks own are balanced by COST, not by instance count: canonical k-mers are twice as dense at the
  // low end of k-mer space as on average and thin out to nothing at the high end, so with equal instance counts the
  // last rank gets five times the buckets of the first -- and a bucket costs the per-bucket kernel as much as ~2100 keys
  // whatever it holds (profiles/r02_local3_experiments.txt): at 8 ranks the last rank's counting took 1.6x the average
  // and everybody waited for it in the final all-reduce.  cost(bucket) = keys + bucket_cost per fine bucket.
  uint32_t bucket_cost = std::is_same<ElemB, uint32_t>::value ? 800u : 0u;   // ~9 ns per bucket over ~12 ps per key (gather + counting)
  if (const char* e = getenv("APGK_BUCKET_COST")) bucket_cost = (uint32_t)std::max(0, atoi(e));
  if (world == 1) bucket_cost = 0;
  const HostLayout hl(world, bins0);
  uint64_t N_sum = 0, N_max = 0;
  for (int s = 0; s < world; s++) { N_sum += meta[s].n_windows; N_max = std::max<uint64_t>(N_max, meta[s].n_windows); }

  // ---- prologue on every local context
  for (RankState& r : g->rs) {
    apgk_ctx* c = r.c;
    GCU(cudaSetDevice(c->device));
    invalidate_results(c);
    stages_reset(c);
    if (!c->res_host) GCU(cudaHostAlloc((void**)&c->res_host, RES_WORDS * 8, cudaHostAllocDefault));
    GCU(c->res.ensure(RES_WORDS * 8));
    GCU(cudaMemsetAsync(c->res.p, 0, RES_WORDS * 8, c->stream));
    if (r.host_words < hl.words) {
      if (r.host) cudaFreeHost(r.host);
      r.host = nullptr; r.host_words = 0;
      GCU(cudaHostAlloc((void**)&r.host, hl.words * 8, cudaHostAllocDefault));
      r.host_words = hl.words;
    }
    r.geom_part = gp;
    r.geom_shard = gp; r.geom_shard.D1 += d2; r.geom_shard.REM -= d2;
    r.nb = nb; r.nbf = nbf;
    r.n_prev = 0; r.shard_n = 0; r.remote_bytes = 0;
    c->geom = gp;
    c->elem_bytes = sizeof(ElemB);
    c->local_max = (uint32_t)local_max;
    c->nb1 = nb;
    c->n_rounds = 0; c->n_big = 0; c->n_distinct = 0; c->n_instances = 0;
    c->table_pending = false;
    c->n_windows_run = c->n_windows;
    stage_begin(c, ST_TOTAL);
    GCU(c->spec_dense.ensure((size_t)SPEC_DENSE * 8));
    GCU(cudaMemsetAsync(c->spec_dense.p, 0, (size_t)SPEC_DENSE * 8, c->stream));
    GCU(c->spec_ovf.ensure(std::max<size_t>((size_t)N_sum / SPEC_DENSE + 16, OVF_SHIP + 2) * 8));
    GCU(cudaMemsetAsync(c->spec_ovf.p, 0, 8, c->stream));
    GCU(c->out_off.ensure(((size_t)nbf + 1) * 8));
    GCU(cudaMemsetAsync(c->out_off.p, 0, ((size_t)nbf + 1) * 8, c->stream));
    GCU(c->nd.ensure(((size_t)nbf + 1) * 4));
    GCU(c->out_off_local.ensure(((size_t)nbf + 1) * 8));
    GCU(c->segtot.ensure((size_t)nbf * 8));
    GCU(c->bofs.ensure(((size_t)nbf + 1) * 8));
    GCU(c->stats.ensure(64));
    GCU(r.sizes32.ensure((size_t)nb * 4));
    GCU(r.sizes_all.ensure((size_t)world * nb * 4));
    GCU(r.tot32.ensure((size_t)nb * 4));
    GCU(r.E_tot.ensure(((size_t)nb + 1) * 8));
    if (bucket_cost) { GCU(r.cost32.ensure((size_t)nb * 4)); GCU(r.E_cost.ensure(((size_t)nb + 1) * 8)); }
    GCU(r.plan_dev.ensure(3 * ((size_t)world + 1) * 8));
    GCU(c->piece_off.ensure((size_t)world * ((size_t)nb + 1) * 8));
    GCU(r.ptrs_dev.ensure(3 * (size_t)world * 8));
    GCU(r.red_in.ensure(((size_t)SPEC_DENSE + 2) * 8));
    GCU(r.red_out.ensure(((size_t)SPEC_DENSE + 2) * 8));
    GCU(r.ovf_all.ensure((size_t)world * (1 + OVF_SHIP) * 8));
    GCU(r.tot0_red.ensure((size_t)bins0 * 8));
  }

  // ---- level-0 histogram on every rank (all rounds share it)
  DigitSpec ds0{DIGIT_BITS, gp.TB - gp.D0, gp.D0, gp.pad, 0};
  DigitFn<DIGIT_BITS> dg0 = make_digit_fn<DIGIT_BITS>(ds0);
  for (RankState& r : g->rs) {
    apgk_ctx* c = r.c;
    GCU(cudaSetDevice(c->device));
    if (c->n_windows) GCTX(c, level0_hist<W>(c, nullptr, 0, dg0));
    else {   // a rank without k-mers still takes part in every collective
      GCTX(c, wait_ingest(c));
      GCU(c->tot0_dev.ensure((size_t)bins0 * 8));
      GCU(cudaMemsetAsync(c->tot0_dev.p, 0, (size_t)bins0 * 8, c->stream));
    }
  }

  // ---- rounds: the same on every rank, cut from the per-bucket MAXIMUM over the ranks
  std::vector<GRound> rounds;
  std::vector<uint64_t> tmax((size_t)bins0, 0);
  if (single) {
    GRound r0{0, bins0, {}};
    r0.inner.push_back({0, bins0});
    rounds.push_back(r0);
  } else {
    { int rc = coll_allreduce_u64(g, (uint64_t)bins0, true, [&](int i) { return (const void*)g->rs[i].c->tot0_dev.p; },
                                  [&](int i) { return (void*)g->rs[i].tot0_red.p; }); if (rc) return rc; }
    for (RankState& r : g->rs) {
      apgk_ctx* c = r.c;
      GCU(cudaSetDevice(c->device));
      GCU(cudaMemcpyAsync(r.host + hl.tot0, c->tot0_dev.p, (size_t)bins0 * 8, cudaMemcpyDeviceToHost, c->stream));
      GCU(cudaMemcpyAsync(r.host + hl.tot0 + bins0, r.tot0_red.p, (size_t)bins0 * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    for (RankState& r : g->rs) {
      GCU(cudaSetDevice(r.c->device));
      GCU(cudaStreamSynchronize(r.c->stream));
      r.tot0.assign(r.host + hl.tot0, r.host + hl.tot0 + bins0);
    }
    for (int d = 0; d < bins0; d++) {
      tmax[d] = g->rs[0].host[hl.tot0 + bins0 + d];
      if (tmax[d] >= (1ull << 32)) GFAIL(APGK_E_RANGE, "level-0 bucket %d holds %llu k-mers on one rank (>= 2^32)", d, (unsigned long long)tmax[d]);
    }
    if (!cap_outer) {
      // Sizes of the rounds from the memory budget: the fewest outer rounds (each is one more pass over the reads)
      // whose level-0 keys leave room for inner rounds of at least a sixteenth of an outer round.
      uint64_t tsum = 0;
      for (int d = 0; d < bins0; d++) tsum += tmax[d];
      const double eA = (double)sizeof(Key<W>);
      budget = (uint64_t)((double)budget * (0.55 / 0.70));   // in rounds the table grows beside the temp buffers: leave it more room
      for (uint64_t ro = 1;; ro++) {
        const double per_outer = (double)tsum / (double)ro * 1.05 + (double)(tsum / (uint64_t)bins0) * 2.0;   // greedy cuts overshoot by a bucket
        const double left = (double)budget - eA * per_outer;
        if (left >= inner_bytes * per_outer / 16.0 || ro >= 64) {
          cap_outer = (uint64_t)std::max(1.0, per_outer);
          cap_inner = cap_inner ? cap_inner : (uint64_t)std::max(1.0, std::min(per_outer, left / inner_bytes));
          break;
        }
      }
    }
    int lo = 0; uint64_t acc = 0;
    auto close_outer = [&](int hi) {
      GRound r{lo, hi, {}};
      int ilo = lo; uint64_t iacc = 0;
      for (int d = lo; d < hi; d++) {
        if (iacc && iacc + tmax[d] > cap_inner) { r.inner.push_back({ilo, d}); ilo = d; iacc = 0; }
        iacc += tmax[d];
      }
      r.inner.push_back({ilo, hi});
      rounds.push_back(r);
    };
    for (int d = 0; d < bins0; d++) {
      if (acc && acc + tmax[d] > cap_outer) { close_outer(d); lo = d; acc = 0; }
      acc += tmax[d];
    }
    close_outer(bins0);
  }
  uint32_t n_inner = 0;
  for (const GRound& r : rounds) n_inner += (uint32_t)r.inner.size();
  auto range_sum = [&](const std::vector<uint64_t>& t, int lo, int hi) { uint64_t s = 0; for (int d = lo; d < hi; d++) s += t[d]; return s; };

  // ---- exported buffers: large enough for every round of this step, then (re)mapped where needed
  {
    std::vector<uint64_t> need_B(world, 0);
    if (single) for (int s = 0; s < world; s++) need_B[s] = meta[s].n_windows * sizeof(ElemB) + 16;
    else {
      uint64_t mx = 0;
      for (const GRound& r : rounds) for (const auto& in : r.inner) mx = std::max(mx, range_sum(tmax, in[0], in[1]));
      for (int s = 0; s < world; s++) need_B[s] = mx * sizeof(ElemB) + 16;
    }
    int rc = refresh_exports(g, meta, need_B, ((uint64_t)nb << d2) * 4 + 16);
    if (rc) return rc;
  }
  for (int i = 0; i < nl; i++) {   // the peers' pointers, for the gather kernels of this step
    RankState& r = g->rs[i];
    apgk_ctx* c = r.c;
    GCU(cudaSetDevice(c->device));
    GCU(cudaMemcpyAsync(r.ptrs_dev.p, r.peer_B.data(), (size_t)world * 8, cudaMemcpyHostToDevice, c->stream));
    GCU(cudaMemcpyAsync(r.ptrs_dev.as<unsigned char>() + (size_t)world * 8, r.peer_sub.data(), (size_t)world * 8, cudaMemcpyHostToDevice, c->stream));
  }

  // ---- the rounds
  bool first_exchange = true;
  std::vector<std::array<uint32_t, 3>> segs;   // ownership of every inner round (host bookkeeping for the lookups)
  for (const GRound& R : rounds) {
    for (RankState& r : g->rs) {
      apgk_ctx* c = r.c;
      GCU(cudaSetDevice(c->device));
      const uint64_t n_o = single ? c->n_windows : range_sum(r.tot0, R.lo, R.hi);
      c->geom = r.geom_part; c->nb1 = nb;
      if (n_o) GCTX(c, level0_scatter<W>(c, nullptr, dg0, R.lo, R.hi, n_o));
    }
    for (const auto& in : R.inner) {
      const int s_lo = in[0], s_hi = in[1];
      // -- this rank's partition of the range; its bucket sizes as u32
      if (!first_exchange) { int rc = coll_barrier_dev(g); if (rc) return rc; }   // the peers are done reading B
      first_exchange = false;
      for (RankState& r : g->rs) {
        apgk_ctx* c = r.c;
        GCU(cudaSetDevice(c->device));
        c->geom = r.geom_part; c->nb1 = nb;
        const uint64_t n_in = single ? c->n_windows : range_sum(r.tot0, s_lo, s_hi);
        const uint64_t off_a = single ? 0 : range_sum(r.tot0, R.lo, s_lo);
        if (n_in) GCTX(c, (level1<W, ElemB>(c, s_lo, s_hi, n_in, c->A.as<Key<W>>() + off_a, d2)));
        else {
          GCU(cudaMemsetAsync(c->segtot.p, 0, (size_t)nb * 8, c->stream));
          GCU(cudaMemsetAsync(c->sub_sizes.p, 0, ((size_t)nb << d2) * 4, c->stream));
        }
        stage_begin(c, ST_PLAN);
        k_sizes32<<<(nb + 255) / 256, 256, 0, c->stream>>>(c->segtot.as<unsigned long long>(), nb, r.sizes32.as<uint32_t>(),
                                                         c->res.as<unsigned long long>() + RES_XFLAGS);
        c->launches++;
        GCU(cudaGetLastError());
      }
      // -- every rank learns every rank's bucket sizes
      { int rc = coll_allgather_dev(g, (size_t)nb * 4, [&](int i) { return (const void*)g->rs[i].sizes32.p; },
                                    [&](int i) { return (void*)g->rs[i].sizes_all.p; }); if (rc) return rc; }
      // -- balanced ranges, offsets of the pieces, one small block to the host
      for (int i = 0; i < nl; i++) {
        RankState& r = g->rs[i];
        apgk_ctx* c = r.c;
        const int me = g->rank0 + i;
        GCU(cudaSetDevice(c->device));
        unsigned long long* flags = c->res.as<unsigned long long>() + RES_XFLAGS;
        k_total_sizes<<<(nb + 255) / 256, 256, 0, c->stream>>>(r.sizes_all.as<uint32_t>(), (uint32_t)world, nb, r.tot32.as<uint32_t>(), flags,
                                                             bucket_cost ? r.cost32.as<uint32_t>() : nullptr, bucket_cost << d2);
        c->launches++;
        GCTX(c, scan_u32(c, r.tot32.as<uint32_t>(), nb, r.E_tot.as<unsigned long long>(), nullptr));
        if (bucket_cost) GCTX(c, scan_u32(c, r.cost32.as<uint32_t>(), nb, r.E_cost.as<unsigned long long>(), nullptr));
        for (int s = 0; s < world; s++)
          GCTX(c, scan_u32(c, r.sizes_all.as<uint32_t>() + (size_t)s * nb, nb,
                           c->piece_off.as<unsigned long long>() + (size_t)s * ((size_t)nb + 1), nullptr));
        k_splitters<<<(world + 1 + 63) / 64, 64, 0, c->stream>>>((bucket_cost ? r.E_cost : r.E_tot).as<unsigned long long>(),
                                                              r.E_tot.as<unsigned long long>(), nb, (uint32_t)world,
                                                              c->piece_off.as<unsigned long long>() + (size_t)me * ((size_t)nb + 1),
                                                              r.plan_dev.as<unsigned long long>());
        c->launches++;
        GCU(cudaGetLastError());
        GCU(cudaMemcpyAsync(r.host + hl.plan, r.plan_dev.p, 3 * ((size_t)world + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
        GCU(cudaMemcpyAsync(r.host + hl.extra, flags, 8, cudaMemcpyDeviceToHost, c->stream));
      }
      // -- the step's one mid-way round trip: the shard's size decides its buffers
      for (int i = 0; i < nl; i++) {
        RankState& r = g->rs[i];
        apgk_ctx* c = r.c;
        const int me = g->rank0 + i;
        GCU(cudaSetDevice(c->device));
        GCU(cudaStreamSynchronize(c->stream));
        stage_end(c, ST_PLAN);
        if (r.host[hl.extra] & 1ull) GFAIL(APGK_E_RANGE, "a bucket piece holds 2^31 or more k-mers");
        if (r.host[hl.extra] & 2ull) GFAIL(APGK_E_RANGE, "a merged bucket holds 2^32 or more k-mers");
        uint32_t lo = (uint32_t)r.host[hl.plan + me], hi = (uint32_t)r.host[hl.plan + me + 1];
        const uint64_t e_lo = r.host[hl.plan + world + 1 + me], e_hi = r.host[hl.plan + world + 1 + me + 1];
        const uint64_t Nr = e_hi - e_lo;
        // only the round's level-0 buckets hold anything: the first and the last rank's ranges reach to the ends
        // of the bucket space, and walking those empty buckets costs more than counting the full ones
        lo = std::max<uint32_t>(lo, (uint32_t)s_lo * (uint32_t)bins1);
        hi = std::min<uint32_t>(hi, (uint32_t)s_hi * (uint32_t)bins1);
        if (hi < lo) hi = lo;
        if (i == 0)   // the bounds are the same on every rank: every rank's clamped range of this inner round
          for (int s = 0; s < world; s++) {
            const uint32_t a = std::max<uint32_t>((uint32_t)r.host[hl.plan + s], (uint32_t)s_lo * (uint32_t)bins1);
            const uint32_t b = std::min<uint32_t>((uint32_t)r.host[hl.plan + s + 1], (uint32_t)s_hi * (uint32_t)bins1);
            if (b > a) segs.push_back({a, b, (uint32_t)s});
          }
        // the gathered shard, the per-bucket records (over the dead level-0 keys when everything ran at once)
        GCU(c->C2.ensure(std::max<uint64_t>(Nr, 1) * sizeof(ElemB) + 16));
        Key<W>* tmp_keys;
        if (single) { GCU(c->A.ensure(std::max<uint64_t>(Nr, 1) * sizeof(Key<W>))); tmp_keys = c->A.as<Key<W>>(); }
        else { GCU(c->TK.ensure(std::max<uint64_t>(Nr, 1) * sizeof(Key<W>))); tmp_keys = c->TK.as<Key<W>>(); }
        stage_begin(c, ST_OWNER);
        GCU(cudaMemsetAsync(c->segtot.p, 0, (size_t)nbf * 8, c->stream));
        GCU(cudaMemsetAsync(c->bofs.p, 0, ((size_t)nbf + 1) * 8, c->stream));
        if (Nr && hi > lo) {
          GatherArgs<ElemB> ga{};
          ga.src_base = (const ElemB* const*)r.ptrs_dev.p; ga.seg_off = nullptr;
          ga.piece_off = c->piece_off.as<unsigned long long>(); ga.sizes_all = r.sizes_all.as<uint32_t>();
          ga.bofs_coarse = r.E_tot.as<unsigned long long>(); ga.coarse_base = e_lo;
          ga.n_src = (uint32_t)world; ga.nb = nb; ga.lo = lo; ga.hi = hi; ga.d2 = d2; ga.digit_pos = gp.REM - d2;
          ga.out = c->C2.as<ElemB>(); ga.bsize_fine = c->segtot.as<unsigned long long>(); ga.bofs_fine = c->bofs.as<unsigned long long>();
          ga.sub_sizes = nullptr;
          ga.sub_ptrs = d2 > 0 ? (const uint32_t* const*)(r.ptrs_dev.as<unsigned char>() + (size_t)world * 8) : nullptr;
          // Two gather kernels, both tested: the direct one (16-byte loads straight from the peers, one in flight per
          // lane) and the one pipelined through shared memory with cp.async (APGK_GATHER=pipelined).  Measured at 8
          // GPUs (profiles/r02_final_bench_n8*.json): 476 against 440 GB/s of remote reads -- with 40+ warps per SM the
          // direct loads already keep the link busy, and the staging costs an extra trip through shared memory.
          const char* eg = getenv("APGK_GATHER");
          const bool direct = !(eg && !strcmp(eg, "pipelined"));
          if (direct) {
            const uint32_t grid = std::min<uint32_t>((hi - lo + 7) / 8, (uint32_t)c->n_sm * 8);  // one warp per bucket
            k_gather_split<ElemB, 256><<<grid, 256, 0, c->stream>>>(ga);
          } else {
            auto kern = k_gather_split2<ElemB, 256>;
            const size_t smg = (size_t)8 * 2 * GsChunk<ElemB>::N * sizeof(ElemB);
            int occ = 1;
            GCTX(c, kernel_setup(c, kern, 256, smg, &occ));
            const uint32_t grid = std::min<uint32_t>((hi - lo + 7) / 8, (uint32_t)c->n_sm * (uint32_t)occ);
            kern<<<grid, 256, smg, c->stream>>>(ga);
          }
          c->launches++;
          GCU(cudaGetLastError());
        }
        stage_end(c, ST_OWNER);
        // -- count the shard: the context now describes the finer geometry (P + d2 prefix bits)
        c->geom = r.geom_shard; c->nb1 = nbf;
        c->n_rounds++;
        r.shard_n += Nr;
        if (Nr && hi > lo) {
          c->count_src = c->C2.p;
          c->bucket_lo = lo << d2; c->bucket_hi = hi << d2;
          c->table_scale = single ? 1.0 : std::max(1.0, (double)N_sum / (double)world / (double)r.shard_n);
          GCTX(c, (count_buckets<W, ElemB>(c, Nr, N_sum, r.n_prev, tmp_keys, single)));
          c->table_scale = 1.0;
          c->bucket_lo = c->bucket_hi = 0;
        }
        // (measurement aid for the single-process form: one rank's shard-side kernels at a time, so that the stage
        // times of contexts that share a device are each rank's own cost -- tools/skew_probe.py)
        static const bool serial = getenv("APGK_GROUP_SERIAL") != nullptr;
        if (serial && !g->use_nccl) GCU(cudaStreamSynchronize(c->stream));
        // bytes this rank's gather pulled from the peers: everything but its own piece
        const uint64_t own = r.host[hl.plan + 2 * (world + 1) + me + 1] - r.host[hl.plan + 2 * (world + 1) + me];
        r.remote_bytes += (Nr - own) * sizeof(ElemB);
      }
    }
  }

  // ---- spectra and totals: one all-reduce (and the barrier that lets the peers reuse their partition buffers)
  for (RankState& r : g->rs) {
    apgk_ctx* c = r.c;
    GCU(cudaSetDevice(c->device));
    stage_begin(c, ST_REDUCE);
    unsigned long long* in = r.red_in.as<unsigned long long>();
    GCU(cudaMemcpyAsync(in, c->spec_dense.p, (size_t)SPEC_DENSE * 8, cudaMemcpyDeviceToDevice, c->stream));
    const unsigned long long ni = r.shard_n;
    GCU(cudaMemcpyAsync(in + SPEC_DENSE, &ni, 8, cudaMemcpyHostToDevice, c->stream));
    if (c->table_pending) GCU(cudaMemcpyAsync(in + SPEC_DENSE + 1, c->res.as<unsigned long long>() + RES_DISTINCT, 8, cudaMemcpyDeviceToDevice, c->stream));
    else { const unsigned long long nd = r.n_prev; GCU(cudaMemcpyAsync(in + SPEC_DENSE + 1, &nd, 8, cudaMemcpyHostToDevice, c->stream)); }
  }
  { int rc = coll_allreduce_u64(g, (uint64_t)SPEC_DENSE + 2, false, [&](int i) { return (const void*)g->rs[i].red_in.p; },
                                [&](int i) { return (void*)g->rs[i].red_out.p; }); if (rc) return rc; }
  // counts beyond the dense range are rare: every rank ships its first OVF_SHIP of them (and how many it has)
  { int rc = coll_allgather_dev(g, (size_t)(1 + OVF_SHIP) * 8, [&](int i) { return (const void*)g->rs[i].c->spec_ovf.p; },
                                [&](int i) { return (void*)g->rs[i].ovf_all.p; }); if (rc) return rc; }
  for (RankState& r : g->rs) {
    apgk_ctx* c = r.c;
    GCU(cudaSetDevice(c->device));
    GCU(cudaMemcpyAsync(r.host + hl.red, r.red_out.p, ((size_t)SPEC_DENSE + 2) * 8, cudaMemcpyDeviceToHost, c->stream));
    GCU(cudaMemcpyAsync(r.host + hl.ovf, r.ovf_all.p, (size_t)world * (1 + OVF_SHIP) * 8, cudaMemcpyDeviceToHost, c->stream));
    stage_end(c, ST_REDUCE);
    stage_end(c, ST_TOTAL);
  }
  for (RankState& r : g->rs) {
    apgk_ctx* c = r.c;
    GCU(cudaSetDevice(c->device));
    GCTX(c, step_epilogue(c, true));          // the step's final synchronisation
    if (!single) c->n_distinct = r.n_prev;
    else if (!c->n_distinct) c->n_distinct = r.n_prev;
    c->n_instances = r.shard_n;
    c->have_table = want_table != 0;
    c->finished = true;
    c->part_ready = false; c->spec_loaded = false; c->table_from_reads = false;
    stages_collect(c);
  }
  // ---- global results (identical on every rank)
  {
    RankState& r = g->rs[0];
    const unsigned long long* red = r.host + hl.red;
    g->sparse_f.clear(); g->sparse_n.clear();
    for (uint64_t f = 1; f < SPEC_DENSE; f++)
      if (red[f]) { g->sparse_f.push_back(f); g->sparse_n.push_back(red[f]); }
    g->n_instances = red[SPEC_DENSE]; g->n_distinct = red[SPEC_DENSE + 1];
    std::vector<uint64_t> far;
    uint64_t worst = 0;
    for (int s = 0; s < world; s++) {
      const unsigned long long* o = r.host + hl.ovf + (size_t)s * (1 + OVF_SHIP);
      worst = std::max<uint64_t>(worst, o[0]);
      for (uint64_t i = 0; i < std::min<uint64_t>(o[0], OVF_SHIP); i++) far.push_back(o[1 + i]);
    }
    if (worst > OVF_SHIP) {
      // more k-mers with counts >= 65536 than the first gather carries: gather the lists at full length
      far.clear();
      const size_t words = 1 + (size_t)worst;
      for (RankState& q : g->rs) { GCU(cudaSetDevice(q.c->device)); GCU(q.ovf_all.ensure((size_t)world * words * 8)); GCU(q.c->spec_ovf.ensure(words * 8)); }
      { int rc = coll_allgather_dev(g, words * 8, [&](int i) { return (const void*)g->rs[i].c->spec_ovf.p; },
                                    [&](int i) { return (void*)g->rs[i].ovf_all.p; }); if (rc) return rc; }
      std::vector<unsigned long long> all((size_t)world * words);
      GCU(cudaSetDevice(r.c->device));
      GCU(cudaMemcpyAsync(all.data(), r.ovf_all.p, all.size() * 8, cudaMemcpyDeviceToHost, r.c->stream));
      for (RankState& q : g->rs) { GCU(cudaSetDevice(q.c->device)); GCU(cudaStreamSynchronize(q.c->stream)); }
      for (int s = 0; s < world; s++)
        for (uint64_t i = 0; i < all[(size_t)s * words]; i++) far.push_back(all[(size_t)s * words + 1 + i]);
    }
    std::sort(far.begin(), far.end());
    for (size_t i = 0; i < far.size();) {
      size_t j = i;
      while (j < far.size() && far[j] == far[i]) j++;
      g->sparse_f.push_back(far[i]); g->sparse_n.push_back(j - i);
      i = j;
    }
    // stats of the first local rank
    apgk_ctx* c = r.c;
    g->stats.world = world; g->stats.n_rounds = (int32_t)n_inner; g->stats.n_outer_rounds = (int32_t)rounds.size();
    g->stats.prefix_bits = gp.D0 + gp.D1; g->stats.split_bits = d2; g->stats.peer_exchange = 1;
    g->stats.shard_instances = r.shard_n;
    g->stats.remote_bytes = r.remote_bytes;
    g->stats.gather_ms = c->stage_ms[ST_OWNER];
    g->stats.step_ms = c->stage_ms[ST_TOTAL];
  }
  std::sort(segs.begin(), segs.end());
  uint32_t covered = 0;
  for (const auto& sg : segs) {
    if (sg[0] != covered) GFAIL(APGK_E_RANGE, "ownership segments do not tile the bucket space (gap or overlap at bucket %u)", covered);
    covered = sg[1];
  }
  if (covered != nb) GFAIL(APGK_E_RANGE, "ownership segments end at bucket %u of %u", covered, nb);
  g->own_segs = segs;
  g->freq_ready = want_table != 0;
  for (RankState& r : g->rs) r.gen_counted = r.c->gen;
  g->counted = true;
  return APGK_OK;
}

int group_count(apgk_group* g) {
  const int world = g->world, nl = g->n_local;
  g->counted = false;
  if (g->dead) GFAIL(APGK_E_STATE, "a context of this group has been destroyed");
  // ---- what every rank tells the others
  std::vector<GroupMeta> mine(nl), meta(world);
  for (int i = 0; i < nl; i++) {
    apgk_ctx* c = g->rs[i].c;
    GCU(cudaSetDevice(c->device));
    GroupMeta& m = mine[i];
    m = GroupMeta{};
    m.n_windows = c->n_windows;
    m.cap_B = c->B.cap; m.cap_sub = c->sub_sizes.cap;
    m.ptr_B = (uint64_t)(uintptr_t)c->B.p; m.ptr_sub = (uint64_t)(uintptr_t)c->sub_sizes.p;
    m.max_round_keys = c->cfg.max_round_keys; m.max_inner_keys = c->cfg.max_inner_keys;
    if (const char* e = getenv("APGK_ROUND_KEYS")) { if (atoll(e) > 0) m.max_round_keys = (uint64_t)atoll(e); }
    if (const char* e = getenv("APGK_INNER_KEYS")) { if (atoll(e) > 0) m.max_inner_keys = (uint64_t)atoll(e); }
    m.K = c->cfg.K; m.flags = (int32_t)(c->cfg.flags & APGK_WANT_COUNTS); m.prefix_bits = c->cfg.prefix_bits;
    // device memory the temp buffers may take: asked once per store size (the query is not cheap)
    if (c->budget_for != c->n_windows + 1) {
      size_t fr = 0, tot = 0;
      GCU(cudaMemGetInfo(&fr, &tot));
      const size_t held = c->A.cap + c->B.cap + c->T.cap + c->C2.cap + c->TK.cap;
      c->budget_bytes = (uint64_t)((double)(fr + held) * 0.70);
      c->budget_for = c->n_windows + 1;
    }
    m.budget = c->budget_bytes;
    if (const char* e = getenv("APGK_BUDGET_BYTES")) { if (atoll(e) > 0) m.budget = (uint64_t)atoll(e); }   // tests: a small device
  }
  { int rc = coll_allgather_host(g, mine.data(), sizeof(GroupMeta), meta.data()); if (rc) return rc; }
  uint64_t N_max = 0, budget = ~0ull, cap_o = 0, cap_i = 0;
  for (int s = 0; s < world; s++) {
    if (meta[s].K != meta[0].K || meta[s].flags != meta[0].flags || meta[s].prefix_bits != meta[0].prefix_bits)
      GFAIL(APGK_E_ARG, "the contexts of a group must share K, APGK_WANT_COUNTS and prefix_bits (rank %d differs)", s);
    N_max = std::max<uint64_t>(N_max, meta[s].n_windows);
    budget = std::min<uint64_t>(budget, meta[s].budget);
    if (meta[s].max_round_keys) cap_o = cap_o ? std::min<uint64_t>(cap_o, meta[s].max_round_keys) : meta[s].max_round_keys;
    if (meta[s].max_inner_keys) cap_i = cap_i ? std::min<uint64_t>(cap_i, meta[s].max_inner_keys) : meta[s].max_inner_keys;
  }
  // ---- same geometry on every rank: chosen for the fullest rank
  apgk_ctx* c0 = g->rs[0].c;
  bool u32 = false;
  for (int i = 0; i < nl; i++) {
    apgk_ctx* c = g->rs[i].c;
    switch (c->W) {
      case 1: u32 = select_geometry<1>(c, N_max, 0); break;
      case 2: select_geometry<2>(c, N_max, 0); break;
      case 3: select_geometry<3>(c, N_max, 0); break;
    }
  }
  const int W = c0->W;
  int d2 = effective_split_bits(c0, ceil_log2(world));
  while (d2 > 0 && ((size_t)4 << (c0->geom.D1 + d2)) > 160 * 1024) d2--;   // the level-1 histogram keeps 2^(D1+d2) counters in shared memory
  // ---- one round or several?  per instance: full key (A) + two level-1 copies (B, gathered shard) + temp count;
  // in rounds the per-bucket records need their own buffer (A keeps the outer round's keys)
  const uint64_t eA = 8ull * W, eB = u32 ? 4 : 8ull * W, eT = (meta[0].flags ? 4 : 0);
  // a shard may exceed the average: by the balance granularity, and because the ranges are balanced by cost (the
  // rank at the dense end of k-mer space gets fewer, fuller buckets: ~1.2x the average instances at 8 ranks)
  const double slack = world > 1 && u32 ? 1.25 : 1.08;
  bool single;
  uint64_t cap_outer = cap_o, cap_inner = cap_i;
  if (cap_o) {
    if (!cap_inner) cap_inner = cap_outer;
    single = N_max <= cap_outer && N_max <= cap_inner;
  } else {
    // everything at once: the rank's own partition (B) + the shard's level-1 copy, records (over the dead level-0 keys) and counts
    single = (double)N_max * ((double)eB + std::max((double)eA, slack * (double)eA) + slack * (double)(eB + eT)) <= (double)budget;
    if (cap_i && N_max > cap_i) single = false;
    cap_outer = 0;   // several rounds: sized in group_count_typed once the level-0 totals of all ranks are known
  }
  const double inner_bytes = (double)eB + slack * (double)(eB + eA + eT);
  if (W == 1) return u32 ? group_count_typed<1, uint32_t>(g, meta, single, cap_outer, cap_inner, d2, budget, inner_bytes)
                         : group_count_typed<1, Key<1>>(g, meta, single, cap_outer, cap_inner, d2, budget, inner_bytes);
  if (W == 2) return group_count_typed<2, Key<2>>(g, meta, single, cap_outer, cap_inner, d2, budget, inner_bytes);
  return group_count_typed<3, Key<3>>(g, meta, single, cap_outer, cap_inner, d2, budget, inner_bytes);
}

// ---------------------------------------------------------------- frequency lookups on the sharded table
// apgk_group_read_freqs_device; the kernels and the data flow are described in gfreq.cuh.

struct FreqMeta {   // what every rank tells the others before a lookup (all-gathered, host side)
  int32_t status, pad_;   // 0, or the error this rank met while preparing
  uint64_t n_bases, batch_bases, cap_B, cap_sub, ptr_B, ptr_sub;
};

// Everything that can fail on one rank alone is decided here, before the call's first collective, and travels to
// the others in FreqMeta::status: a rank that failed on its own between two collectives would leave the others
// waiting in the next one.
int gfreq_prepare(apgk_group* g, int i, uint32_t* const* d_out, const uint64_t* first_base, const uint64_t* n_bases, FreqMeta& m) {
  RankState& r = g->rs[i];
  apgk_ctx* c = r.c;
  const int me = g->rank0 + i;
  m = FreqMeta{};
  m.cap_B = c->B.cap; m.cap_sub = c->sub_sizes.cap;
  m.ptr_B = (uint64_t)(uintptr_t)c->B.p; m.ptr_sub = (uint64_t)(uintptr_t)c->sub_sizes.p;
  if (!d_out || !first_base || !n_bases) GFAIL(APGK_E_ARG, "apgk_group_read_freqs_device: d_out, first_base and n_bases are required");
  if (!g->counted || !g->freq_ready)
    GFAIL(APGK_E_STATE, "apgk_group_read_freqs_device needs a completed apgk_group_count with APGK_WANT_COUNTS");
  if (c->gen != r.gen_counted)
    GFAIL(APGK_E_STATE, "rank %d: its context was reset, given reads or counted on its own since apgk_group_count: count again", me);
  if (first_base[i] > c->total_bases || n_bases[i] > c->total_bases - first_base[i])
    GFAIL(APGK_E_ARG, "rank %d: bases [%llu, +%llu) lie beyond its read store of %llu bases", me, (unsigned long long)first_base[i],
          (unsigned long long)n_bases[i], (unsigned long long)c->total_bases);
  if (n_bases[i] && !d_out[i]) GFAIL(APGK_E_ARG, "rank %d: no output buffer", me);
  m.n_bases = n_bases[i];
  GCU(cudaSetDevice(c->device));
  // batch size from the budget of the count's temp buffers: per base at most one element in B and one position
  uint64_t budget = c->budget_bytes;
  if (const char* e = getenv("APGK_BUDGET_BYTES")) { if (atoll(e) > 0) budget = (uint64_t)atoll(e); }   // tests: a small device
  const uint64_t eb = c->elem_bytes;
  m.batch_bases = std::min<uint64_t>(std::max<uint64_t>(budget / (eb + 4), 4096), 1ull << 31) & ~15ull;
  const uint64_t per = std::min(m.batch_bases, m.n_bases);
  const uint32_t nb = r.nb;
  const int world = g->world;
  GCU(r.gpos.ensure(std::max<uint64_t>(per, 1) * 4));
  GCU(r.gcnt.ensure(64));
  GCU(c->piece_off.ensure((size_t)world * ((size_t)nb + 1) * 8));
  GCU(r.sizes32.ensure((size_t)nb * 4));
  GCU(r.sizes_all.ensure((size_t)world * nb * 4));
  GCU(c->occ_bcur.ensure((size_t)nb * 8));
  GCU(r.ptrs_dev.ensure(3 * (size_t)world * 8));
  GCU(r.red_out.ensure(64));
  GCU(c->blocksum.ensure((((size_t)nb + 1 + SCAN_BLOCK - 1) / SCAN_BLOCK + 1) * 8));   // what scan_u32 takes
  for (cudaEvent_t& e : r.gev) if (!e) GCU(cudaEventCreate(&e));
  // B grows later, in refresh_exports (peers may have it mapped): here only whether it can
  const uint64_t need_B = per * eb + 16;
  if (need_B > c->B.cap) {
    size_t fr = 0, tot = 0;
    GCU(cudaMemGetInfo(&fr, &tot));
    if ((uint64_t)fr + c->B.cap < need_B + (64ull << 20))
      GFAIL(APGK_E_NOMEM, "rank %d: the partition buffer needs %llu bytes, %llu free", me, (unsigned long long)need_B, (unsigned long long)fr);
  }
  return APGK_OK;
}

template <int W, typename Elem>
int group_read_freqs_typed(apgk_group* g, uint32_t* const* d_out, const uint64_t* first_base, const std::vector<FreqMeta>& meta,
                           apgk_group_freq_stats* st) {
  const int world = g->world, nl = g->n_local;
  constexpr uint64_t eb = sizeof(Elem);
  uint64_t BB = ~0ull, n_batches = 0;
  for (int s = 0; s < world; s++) BB = std::min<uint64_t>(BB, meta[s].batch_bases);
  for (int s = 0; s < world; s++) n_batches = std::max<uint64_t>(n_batches, (meta[s].n_bases + BB - 1) / BB);
  // every rank's B large enough for one batch, re-exported where it grew (after apgk_release_temp too)
  {
    std::vector<GroupMeta> gm(world);
    std::vector<uint64_t> need_B(world);
    for (int s = 0; s < world; s++) {
      gm[s] = GroupMeta{};
      gm[s].cap_B = meta[s].cap_B; gm[s].cap_sub = meta[s].cap_sub; gm[s].ptr_B = meta[s].ptr_B; gm[s].ptr_sub = meta[s].ptr_sub;
      need_B[s] = std::min(BB, meta[s].n_bases) * eb + 16;
    }
    int rc = refresh_exports(g, gm, need_B, 16);
    if (rc) return rc;
  }
  RankState& r0 = g->rs[0];
  apgk_ctx* c0 = r0.c;
  for (RankState& r : g->rs) {
    apgk_ctx* c = r.c;
    GCU(cudaSetDevice(c->device));
    { int rc = wait_ingest(c); if (rc) return rc; }
    GCU(cudaMemcpyAsync(r.ptrs_dev.p, r.peer_B.data(), (size_t)world * 8, cudaMemcpyHostToDevice, c->stream));
    GCU(cudaMemsetAsync(r.gcnt.p, 0, 64, c->stream));
  }
  GCU(cudaSetDevice(c0->device));
  GCU(cudaEventRecord(r0.gev[4], c0->stream));
  float ms[3] = {0, 0, 0};
  auto collect = [&]() {   // stage times of the batch just run, first local context
    cudaEventSynchronize(r0.gev[3]);
    for (int k = 0; k < 3; k++) { float x = 0; if (cudaEventElapsedTime(&x, r0.gev[k], r0.gev[k + 1]) == cudaSuccess) ms[k] += x; }
  };
  constexpr int NT = 128;
  for (uint64_t k = 0; k < n_batches; k++) {
    if (k) collect();
    // -- sender: histogram of the batch's windows by coarse bucket, bucket starts, elements into B
    for (int i = 0; i < nl; i++) {
      RankState& r = g->rs[i];
      apgk_ctx* c = r.c;
      const int me = g->rank0 + i;
      GCU(cudaSetDevice(c->device));
      if (i == 0) GCU(cudaEventRecord(r.gev[0], c->stream));
      const uint32_t nb = r.nb;
      const uint64_t n = meta[me].n_bases, b0 = std::min(k * BB, n), nbb = std::min(BB, n - b0), first = first_base[i] + b0;
      FreqTable<W> tp{};   // the partition geometry: the sweep reads only the bucket digit's position
      tp.prefix_pos = r.geom_part.REM; tp.prefix_len = r.geom_part.D0 + r.geom_part.D1; tp.pad = r.geom_part.pad;
      unsigned long long* own = c->piece_off.as<unsigned long long>() + (size_t)me * ((size_t)nb + 1);
      unsigned long long* cnt = r.gcnt.as<unsigned long long>();
      const unsigned grid = (unsigned)((((first & 15) + nbb + POS_PER_THREAD - 1) / POS_PER_THREAD + NT - 1) / NT);
      GCU(cudaMemsetAsync(r.sizes32.p, 0, (size_t)nb * 4, c->stream));
      if (nbb) {
        GCU(cudaMemsetAsync(d_out[i] + b0, 0xFF, nbb * 4, c->stream));
        k_occ_scatter<W, Elem, uint32_t, NT><<<grid, NT, 0, c->stream>>>(read_store(c), tp, first, nbb, r.sizes32.as<uint32_t>(), nullptr,
                                                                        nullptr, nullptr, 0, 0, cnt);
        c->launches++;
        GCU(cudaGetLastError());
      }
      GCTX(c, scan_u32(c, r.sizes32.as<uint32_t>(), nb, own, nullptr));
      if (nbb) {
        GCU(cudaMemcpyAsync(c->occ_bcur.p, own, (size_t)nb * 8, cudaMemcpyDeviceToDevice, c->stream));
        k_occ_scatter<W, Elem, uint32_t, NT><<<grid, NT, 0, c->stream>>>(read_store(c), tp, first, nbb, nullptr, c->occ_bcur.as<unsigned long long>(),
                                                                        c->B.as<Elem>(), r.gpos.as<uint32_t>(), 0, nbb, cnt);
        c->launches++;
        GCU(cudaGetLastError());
      }
      if (i == 0) GCU(cudaEventRecord(r.gev[1], c->stream));
    }
    // -- every rank learns every rank's bucket sizes (this also orders the owners' reads after the senders' sweeps)
    { int rc = coll_allgather_dev(g, (size_t)g->rs[0].nb * 4, [&](int i) { return (const void*)g->rs[i].sizes32.p; },
                                  [&](int i) { return (void*)g->rs[i].sizes_all.p; }); if (rc) return rc; }
    // -- owner: the pieces of its buckets, resolved in place in the senders' B
    for (int i = 0; i < nl; i++) {
      RankState& r = g->rs[i];
      apgk_ctx* c = r.c;
      const int me = g->rank0 + i;
      const uint32_t nb = r.nb;
      GCU(cudaSetDevice(c->device));
      for (int s = 0; s < world; s++)
        if (s != me)
          GCTX(c, scan_u32(c, r.sizes_all.as<uint32_t>() + (size_t)s * nb, nb, c->piece_off.as<unsigned long long>() + (size_t)s * ((size_t)nb + 1), nullptr));
      FreqTable<W> ts = freq_table<W>(c);   // the shard's table, indexed by the finer bucket of the count (P + d2 bits)
      ts.nb = r.nbf; ts.prefix_pos = r.geom_shard.REM; ts.prefix_len = r.geom_shard.D0 + r.geom_shard.D1; ts.pad = r.geom_shard.pad;
      ts.D1 = r.geom_shard.D1;
      GfArgs<Elem> a{};
      a.src = (Elem* const*)r.ptrs_dev.p; a.piece_off = c->piece_off.as<unsigned long long>();
      a.n_src = (uint32_t)world; a.nb = nb; a.me = (uint32_t)me;
      a.d2 = r.geom_shard.D1 - r.geom_part.D1; a.rem_bits = r.geom_part.REM; a.pad = r.geom_part.pad;
      a.counters = r.gcnt.as<unsigned long long>();
      for (const auto& sg : g->own_segs) {
        if ((int)sg[2] != me) continue;
        a.lo = sg[0]; a.hi = sg[1];
        k_gf_resolve<W, Elem, GF_NT><<<std::min<uint32_t>(sg[1] - sg[0], (uint32_t)c->n_sm * 8), GF_NT, 0, c->stream>>>(ts, a);
        c->launches++;
        GCU(cudaGetLastError());
      }
    }
    // -- all owners are done.  Their stores into this rank's B were made by kernels that had completed when their
    // streams reached the barrier; a kernel's stores, peer stores included, are visible to every device once it has
    // completed, and this rank's scatter runs after the barrier on its stream.  (The barrier also keeps the next
    // batch's sweep from overwriting B while an owner still reads it.)
    { int rc = coll_barrier_dev(g); if (rc) return rc; }
    for (int i = 0; i < nl; i++) {
      RankState& r = g->rs[i];
      apgk_ctx* c = r.c;
      const int me = g->rank0 + i;
      GCU(cudaSetDevice(c->device));
      if (i == 0) GCU(cudaEventRecord(r.gev[2], c->stream));
      const uint64_t n = meta[me].n_bases, b0 = std::min(k * BB, n), nbb = std::min(BB, n - b0);
      if (nbb) {
        const unsigned long long* own = c->piece_off.as<unsigned long long>() + (size_t)me * ((size_t)r.nb + 1);
        k_gf_scatter<Elem><<<(unsigned)std::min<uint64_t>((nbb + 255) / 256, (uint64_t)c->n_sm * 8), 256, 0, c->stream>>>(
            c->B.as<Elem>(), r.gpos.as<uint32_t>(), own + r.nb, d_out[i] + b0, r.gcnt.as<unsigned long long>());
        c->launches++;
        GCU(cudaGetLastError());
      }
      if (i == 0) GCU(cudaEventRecord(r.gev[3], c->stream));
    }
  }
  // windows missing from their owner's table (or beyond their bucket) summed over the ranks: a table that does not
  // match the reads fails the call on every rank
  { int rc = coll_allreduce_u64(g, 4, false, [&](int i) { return (const void*)g->rs[i].gcnt.p; },
                                [&](int i) { return (void*)g->rs[i].red_out.p; }); if (rc) return rc; }
  unsigned long long red[4] = {0, 0, 0, 0}, own[4] = {0, 0, 0, 0};
  GCU(cudaSetDevice(c0->device));
  GCU(cudaEventRecord(r0.gev[5], c0->stream));
  GCU(cudaMemcpyAsync(red, r0.red_out.p, 32, cudaMemcpyDeviceToHost, c0->stream));
  GCU(cudaMemcpyAsync(own, r0.gcnt.p, 32, cudaMemcpyDeviceToHost, c0->stream));
  for (RankState& r : g->rs) { GCU(cudaSetDevice(r.c->device)); GCU(cudaStreamSynchronize(r.c->stream)); }
  if (n_batches) collect();
  if (red[0] || red[2])
    GFAIL(APGK_E_STATE, "group read_freqs: %llu windows missing from their owner's table, %llu beyond their bucket (the tables do not match the reads)",
          red[0], red[2]);
  if (st) {
    *st = apgk_group_freq_stats{};
    st->n_batches = (int32_t)n_batches;
    st->n_queries = own[3];
    st->remote_bytes = own[1] * (eb + 4);
    st->sweep_ms = ms[0]; st->exchange_ms = ms[1]; st->scatter_ms = ms[2];
    cudaEventElapsedTime(&st->total_ms, r0.gev[4], r0.gev[5]);
  }
  return APGK_OK;
}

int group_read_freqs(apgk_group* g, uint32_t* const* d_out, const uint64_t* first_base, const uint64_t* n_bases, apgk_group_freq_stats* st) {
  if (g->dead) GFAIL(APGK_E_STATE, "a context of this group has been destroyed");
  const int world = g->world, nl = g->n_local;
  std::vector<FreqMeta> mine(nl), meta(world);
  std::string own_err;
  for (int i = 0; i < nl; i++) {
    const int rc = gfreq_prepare(g, i, d_out, first_base, n_bases, mine[i]);
    if (rc) { mine[i].status = rc; if (own_err.empty()) own_err = g->err; }
  }
  { int rc = coll_allgather_host(g, mine.data(), sizeof(FreqMeta), meta.data()); if (rc) return rc; }
  for (int s = 0; s < world; s++)
    if (meta[s].status) {
      if (own_err.empty()) GFAIL(meta[s].status, "rank %d refused the lookup (error %d; its apgk_group_last_error says why)", s, meta[s].status);
      g->err = own_err;
      return meta[s].status;
    }
  apgk_ctx* c0 = g->rs[0].c;
  if (c0->elem_bytes == 4) return group_read_freqs_typed<1, uint32_t>(g, d_out, first_base, meta, st);
  if (c0->W == 1) return group_read_freqs_typed<1, Key<1>>(g, d_out, first_base, meta, st);
  if (c0->W == 2) return group_read_freqs_typed<2, Key<2>>(g, d_out, first_base, meta, st);
  return group_read_freqs_typed<3, Key<3>>(g, d_out, first_base, meta, st);
}

}  // namespace
