// C++ host test of the frequency lookups on the sharded table (apgk_group_read_freqs_device, include/apgk.h), without
// Python or torch.
//
//   test_group_freqs local N   one process, N contexts on device 0 (apgk_group_local): runs on a one-GPU box
//   test_group_freqs procs N   N processes, one GPU each (NCCL + CUDA IPC, as tests/cpp/test_group.cpp); exits 77
//                              ("skipped") when the box has fewer than N GPUs
//
// Each rank generates its slice of one synthetic read set, the group counts it and every rank looks up the global
// count of every window of its reads; the concatenated answers must equal apgk_read_freqs of ONE context over all
// the reads.  A lookup over a sub-range (unaligned, empty on one rank) follows.  Prints "FREQS OK" on success.
#include <unistd.h>
#include <sys/wait.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "apgk.h"

#define REQUIRE(c) do { if (!(c)) { std::fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #c); return 1; } } while (0)
#define OK(call) do { int rc__ = (call); if (rc__ != APGK_OK) { std::fprintf(stderr, "FAILED %s:%d: %s -> %d\n", __FILE__, __LINE__, #call, rc__); return 1; } } while (0)

static const int K = 25;
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
// the single-GPU answer over reads [0, n_total): the count at every base
static int reference_freqs(int device, uint64_t genome, uint64_t n_total, std::vector<uint32_t>& out) {
  apgk_ctx* c = nullptr;
  OK(make_ctx(device, &c));
  apgk_synth_params sp = synth(genome);
  OK(apgk_synth_reads(c, &sp, 0, n_total));
  OK(apgk_finish(c));
  uint64_t tb = 0, nr = 0;
  OK(apgk_read_store_info(c, &tb, &nr));
  out.resize(tb);
  OK(apgk_read_freqs(c, 0, tb, out.data()));
  apgk_destroy(c);
  return 0;
}
// ranks' lookups of [first[j], first[j] + n[j]) of their stores (rank r's store = reference bases [r * per, ...))
static int lookup_and_check(apgk_group* g, std::vector<apgk_ctx*>& cs, int rank0, uint64_t per, const std::vector<uint64_t>& first,
                            const std::vector<uint64_t>& n, const std::vector<uint32_t>& ref) {
  const int nl = (int)cs.size();
  std::vector<uint32_t*> d(nl, nullptr);
  for (int j = 0; j < nl; j++) OK(apgk_device_alloc(cs[j], (void**)&d[j], (n[j] ? n[j] : 1) * 4));
  apgk_group_freq_stats st;
  if (apgk_group_read_freqs_device(g, d.data(), first.data(), n.data(), &st) != APGK_OK) {
    std::fprintf(stderr, "apgk_group_read_freqs_device: %s\n", apgk_group_last_error(g));
    return 1;
  }
  REQUIRE(st.n_batches >= 1 && st.total_ms > 0);
  for (int j = 0; j < nl; j++) {
    std::vector<uint32_t> h(n[j]);
    if (n[j]) OK(apgk_device_copy_to_host(cs[j], h.data(), d[j], n[j] * 4));
    const uint64_t base = (uint64_t)(rank0 + j) * per + first[j];
    for (uint64_t i = 0; i < n[j]; i++)
      if (h[i] != ref[base + i]) { std::fprintf(stderr, "rank %d base %llu: %u != %u\n", rank0 + j, (unsigned long long)(first[j] + i), h[i], ref[base + i]); return 1; }
    OK(apgk_device_free(cs[j], d[j]));
  }
  return 0;
}

static int run_ranks(apgk_group* g, std::vector<apgk_ctx*>& cs, int rank0, uint64_t per_bases, const std::vector<uint32_t>& ref) {
  const int nl = (int)cs.size();
  if (apgk_group_count(g) != APGK_OK) { std::fprintf(stderr, "apgk_group_count: %s\n", apgk_group_last_error(g)); return 1; }
  std::vector<uint64_t> first(nl, 0), n(nl, per_bases);
  if (lookup_and_check(g, cs, rank0, per_bases, first, n, ref)) return 1;
  for (int j = 0; j < nl; j++) {   // unaligned ranges; rank 1 asks nothing
    first[j] = 17 + j;
    n[j] = (rank0 + j == 1) ? 0 : per_bases - 30 - j;
  }
  return lookup_and_check(g, cs, rank0, per_bases, first, n, ref);
}

static int run_local(int world) {
  const uint64_t genome = 400000, n_per = 30000;
  std::vector<uint32_t> ref;
  if (reference_freqs(0, genome, n_per * world, ref)) return 1;
  std::vector<apgk_ctx*> cs(world, nullptr);
  apgk_synth_params sp = synth(genome);
  for (int r = 0; r < world; r++) { OK(make_ctx(0, &cs[r])); OK(apgk_synth_reads(cs[r], &sp, r * n_per, n_per)); }
  apgk_group* g = nullptr;
  OK(apgk_group_local(cs.data(), world, &g));
  if (run_ranks(g, cs, 0, n_per * 100, ref)) return 1;
  apgk_group_destroy(g);
  for (apgk_ctx* c : cs) apgk_destroy(c);
  std::printf("FREQS OK (single process, %d contexts on one device)\n", world);
  return 0;
}

static int rank_main(int rank, int world, const uint8_t* id) {
  const uint64_t genome = 2000000, n_per = 300000;
  std::vector<uint32_t> ref;
  if (reference_freqs(rank, genome, n_per * world, ref)) return 1;   // every rank computes the whole answer on its own GPU
  std::vector<apgk_ctx*> cs(1, nullptr);
  OK(make_ctx(rank, &cs[0]));
  apgk_synth_params sp = synth(genome);
  OK(apgk_synth_reads(cs[0], &sp, rank * n_per, n_per));
  apgk_group* g = nullptr;
  if (apgk_group_join(cs[0], id, rank, world, &g) != APGK_OK) { std::fprintf(stderr, "rank %d: join: %s\n", rank, apgk_last_error(cs[0])); return 1; }
  if (run_ranks(g, cs, rank, n_per * 100, ref)) return 1;
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
  std::printf("FREQS OK (%d processes, one GPU each, NCCL + CUDA IPC)\n", world);
  return 0;
}

int main(int argc, char** argv) {
  const bool procs = argc > 1 && !std::strcmp(argv[1], "procs");
  const int world = argc > 2 ? std::atoi(argv[2]) : 3;
  if (world < 2 || world > 16) return 2;
  return procs ? run_procs(world) : run_local(world);
}
