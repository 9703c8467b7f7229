// C++ host test of the occurrence records on the sharded table (apgk_group_build_occurrences, include/apgk.h), without
// Python or torch.
//
//   test_group_occurrences local N   one process, N contexts on device 0 (apgk_group_local): runs on a one-GPU box
//   test_group_occurrences procs N   N processes, one GPU each (NCCL + CUDA IPC, as tests/cpp/test_group.cpp); exits
//                                    77 ("skipped") when the box has fewer than N GPUs
//
// Each rank generates its slice of one synthetic read set (rank r holds reads [r * n, (r + 1) * n), so group read ids
// are the read set's own numbers), the group counts it and builds the records; every row of every shard must equal
// the row of the same k-mer in ONE context's apgk_build_occurrences over all the reads (count, read ids and signed
// positions), and the shards together hold all of its instances.  Prints "OCCURRENCES OK" on success.
#include <unistd.h>
#include <sys/wait.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "apgk.h"

#define REQUIRE(c) do { if (!(c)) { std::fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #c); return 1; } } while (0)
#define OK(call) do { int rc__ = (call); if (rc__ != APGK_OK) { std::fprintf(stderr, "FAILED %s:%d: %s -> %d\n", __FILE__, __LINE__, #call, rc__); return 1; } } while (0)

static const int K = 25;   // one-word keys
static apgk_synth_params synth(uint64_t genome) {
  apgk_synth_params p{};
  p.genome_len = genome; p.seed_g = 0xA11BA7C5; p.seed_p = 0x5EED00A0; p.seed_q = 0x5EED00A1; p.seed_r = 0x5EED0001; p.seed_e = 0x5EED0002;
  p.read_len = 100; p.err_per_200 = 1;
  return p;
}
static int make_ctx(int device, apgk_ctx** c) {
  apgk_config cfg{};
  cfg.K = K; cfg.device = device; cfg.flags = APGK_WANT_COUNTS;
  return apgk_create(&cfg, c);
}
struct Table { std::vector<uint64_t> keys, run_off; std::vector<uint32_t> counts, read_id; std::vector<int32_t> pos; };
static int table_of(apgk_ctx* c, Table& t) {
  uint64_t ni = 0, nd = 0, n_occ = 0;
  OK(apgk_totals(c, &ni, &nd));
  OK(apgk_occurrences_info(c, &n_occ, nullptr, nullptr));
  REQUIRE(n_occ == ni);
  t.keys.resize(nd); t.counts.resize(nd); t.run_off.resize(nd + 1); t.read_id.resize(ni + 1); t.pos.resize(ni + 1);
  OK(apgk_counts_copy(c, 0, nd, t.keys.data(), t.counts.data()));
  OK(apgk_occurrences_copy(c, 0, nd, t.run_off.data(), t.read_id.data(), t.pos.data()));
  REQUIRE(t.run_off[0] == 0 && t.run_off[nd] == ni);
  return 0;
}
// the single-GPU answer over reads [0, n_total)
static int reference_table(int device, uint64_t genome, uint64_t n_total, Table& ref) {
  apgk_ctx* c = nullptr;
  OK(make_ctx(device, &c));
  apgk_synth_params sp = synth(genome);
  OK(apgk_synth_reads(c, &sp, 0, n_total));
  OK(apgk_finish(c));
  OK(apgk_build_occurrences(c));
  if (table_of(c, ref)) return 1;
  apgk_destroy(c);
  return 0;
}

static int run_ranks(apgk_group* g, std::vector<apgk_ctx*>& cs, int rank0, const Table& ref) {
  if (apgk_group_count(g) != APGK_OK) { std::fprintf(stderr, "apgk_group_count: %s\n", apgk_group_last_error(g)); return 1; }
  uint64_t one = 0;
  REQUIRE(apgk_occurrences_copy(cs[0], 0, 0, &one, nullptr, nullptr) == APGK_E_STATE);   // a shard has none before the group build
  REQUIRE(apgk_build_occurrences(cs[0]) == APGK_E_STATE);                                // nor can it build its own
  apgk_group_occ_stats st;
  if (apgk_group_build_occurrences(g, &st) != APGK_OK) {
    std::fprintf(stderr, "apgk_group_build_occurrences: %s\n", apgk_group_last_error(g));
    return 1;
  }
  REQUIRE(st.n_batches >= 1 && st.n_windows > 0 && st.total_ms > 0);
  uint64_t gi = 0, gd = 0, held = 0;
  OK(apgk_group_totals(g, &gi, &gd));
  REQUIRE(gd == ref.keys.size() && gi == ref.read_id.size() - 1);
  for (size_t j = 0; j < cs.size(); j++) {
    Table t;
    if (table_of(cs[j], t)) return 1;
    if (j == 0) REQUIRE(st.n_occ == t.read_id.size() - 1);
    held += t.read_id.size() - 1;
    for (size_t i = 0; i < t.keys.size(); i++) {
      const auto it = std::lower_bound(ref.keys.begin(), ref.keys.end(), t.keys[i]);
      REQUIRE(it != ref.keys.end() && *it == t.keys[i]);
      const size_t r = (size_t)(it - ref.keys.begin());
      const uint64_t a = t.run_off[i], b = ref.run_off[r], n = ref.run_off[r + 1] - b;
      bool same = t.counts[i] == ref.counts[r] && t.run_off[i + 1] - a == n;
      for (uint64_t k = 0; same && k < n; k++) same = t.read_id[a + k] == ref.read_id[b + k] && t.pos[a + k] == ref.pos[b + k];
      if (!same) {
        std::fprintf(stderr, "rank %d row %zu: count %u, %llu records; one context: count %u, %llu records (or a record differs)\n",
                     rank0 + (int)j, i, t.counts[i], (unsigned long long)(t.run_off[i + 1] - a), ref.counts[r], (unsigned long long)n);
        return 1;
      }
    }
  }
  if (cs.size() > 1) REQUIRE(held == gi);   // in the single-process form this process holds every shard
  return 0;
}

static int run_local(int world) {
  const uint64_t genome = 400000, n_per = 30000;
  Table ref;
  if (reference_table(0, genome, n_per * world, ref)) return 1;
  std::vector<apgk_ctx*> cs(world, nullptr);
  apgk_synth_params sp = synth(genome);
  for (int r = 0; r < world; r++) { OK(make_ctx(0, &cs[r])); OK(apgk_synth_reads(cs[r], &sp, r * n_per, n_per)); }
  apgk_group* g = nullptr;
  OK(apgk_group_local(cs.data(), world, &g));
  if (run_ranks(g, cs, 0, ref)) return 1;
  apgk_group_destroy(g);
  for (apgk_ctx* c : cs) apgk_destroy(c);
  std::printf("OCCURRENCES OK (single process, %d contexts on one device)\n", world);
  return 0;
}

static int rank_main(int rank, int world, const uint8_t* id) {
  const uint64_t genome = 2000000, n_per = 300000;
  Table ref;
  if (reference_table(rank, genome, n_per * world, ref)) return 1;   // every rank computes the whole answer on its own GPU
  std::vector<apgk_ctx*> cs(1, nullptr);
  OK(make_ctx(rank, &cs[0]));
  apgk_synth_params sp = synth(genome);
  OK(apgk_synth_reads(cs[0], &sp, rank * n_per, n_per));
  apgk_group* g = nullptr;
  if (apgk_group_join(cs[0], id, rank, world, &g) != APGK_OK) { std::fprintf(stderr, "rank %d: join: %s\n", rank, apgk_last_error(cs[0])); return 1; }
  if (run_ranks(g, cs, rank, ref)) return 1;
  apgk_group_destroy(g);
  apgk_destroy(cs[0]);
  return 0;
}

static int run_procs(int world) {
  // count the GPUs in a child: the parent must not hold a CUDA context across fork()
  int pfd[2];
  if (pipe(pfd)) return 1;
  pid_t probe = fork();
  if (probe == 0) {
    apgk_ctx* c = nullptr;
    int n = 0;
    while (n < 64 && make_ctx(n, &c) == APGK_OK) { apgk_destroy(c); n++; }
    if (write(pfd[1], &n, sizeof n) != (ssize_t)sizeof n) _exit(1);
    _exit(0);
  }
  int ngpu = 0;
  if (read(pfd[0], &ngpu, sizeof ngpu) != (ssize_t)sizeof ngpu) ngpu = 0;
  waitpid(probe, nullptr, 0);
  if (ngpu < world) { std::printf("SKIPPED: %d GPUs, %d needed\n", ngpu, world); return 77; }
  std::vector<int> rd(world, -1), wr(world, -1);
  for (int r = 1; r < world; r++) { int p[2]; if (pipe(p)) return 1; rd[r] = p[0]; wr[r] = p[1]; }
  std::vector<pid_t> kids;
  for (int r = 0; r < world; r++) {
    pid_t pid = fork();
    if (pid == 0) {
      uint8_t id[APGK_GROUP_ID_BYTES];
      if (r == 0) {
        if (apgk_group_unique_id(id) != APGK_OK) { std::fprintf(stderr, "apgk_group_unique_id failed (libnccl.so.2?)\n"); _exit(1); }
        for (int s = 1; s < world; s++) if (write(wr[s], id, sizeof id) != (ssize_t)sizeof id) _exit(1);
      } else if (read(rd[r], id, sizeof id) != (ssize_t)sizeof id) _exit(1);
      _exit(rank_main(r, world, id));
    }
    kids.push_back(pid);
  }
  int bad = 0;
  for (pid_t k : kids) { int st = 0; waitpid(k, &st, 0); if (!WIFEXITED(st) || WEXITSTATUS(st) != 0) bad++; }
  if (bad) { std::fprintf(stderr, "%d rank(s) failed\n", bad); return 1; }
  std::printf("OCCURRENCES OK (%d processes, one GPU each, NCCL + CUDA IPC)\n", world);
  return 0;
}

int main(int argc, char** argv) {
  const bool procs = argc > 1 && !std::strcmp(argv[1], "procs");
  const int world = argc > 2 ? std::atoi(argv[2]) : 3;
  if (world < 2 || world > 16) return 2;
  return procs ? run_procs(world) : run_local(world);
}
